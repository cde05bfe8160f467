// scan.cu -- parallel-in-time Kalman filter / RTS smoother for ONE long series
// (BASELINE.json config 5; not in the reference, whose time recursion is strictly
// sequential -- Filter.scala:41-62, and whose FilterTs.scanRight is literally `???`).
//
// Formulation: Sarkka & Garcia-Fernandez, "Temporal Parallelization of Bayesian Smoothers"
// (IEEE TAC 2021) mapped to DLM notation (H = F^T, Q = W dt, R = V; SURVEY.md Appendix C).
// Two-level scan, organised for HBM:
//   level 1  every thread owns kSub consecutive time points and composes their filtering
//            elements (A, b, C, eta, J) sequentially, reading only y (8 B / step);
//   level 2  the per-thread aggregates (T / kSub of them, a few MB) are scanned with the
//            associative operator (block-wide Hillis-Steele in shared memory + one
//            recursion over block totals);
//   apply    every thread starts from its exclusive prefix -- whose (b, C) IS the filtered
//            (m, C) at its first time point -- and runs the ordinary sequential Kalman
//            recursion (the same register code as kf_small.cu) over its kSub steps,
//            writing the KfState outputs.  The smoother repeats this backwards with the
//            elements (E, g, L); its apply phase is the sequential RTS step in textbook mode.
// Elements are never materialised per time point: HBM traffic is y twice + outputs once.
// The backward sampler of FFBS (bdlm_scan_ffbs) is a third scan of the same shape, over the affine
// maps theta_r = B_r theta_{r+1} + c_r, with the Gibbs statistics summed in its apply sweep.
//
// Multi-GPU: a rank's chunk aggregate (3n^2+2n doubles forward, 2n^2+n backward, n^2+n for the
// sampler) is all that crosses the fabric (one all-gather per pass), plus one all-gather of the
// rank's partial sums for the log-likelihoods and the Gibbs statistics; the carry is folded on the device.
//
// Parity: equals the sequential kernel in textbook-smoother mode to 1e-9 relative (for n = 1
// that is the reference itself); the apply phases reuse the sequential step code, so the
// only difference is the rounding of the scanned start states.
#include <cmath>
#include <type_traits>
#include <vector>

#include "common.cuh"
#include "launch.h"
#include "rng.cuh"
#include "small_steps.cuh"

namespace bdlm {

using namespace small;

// ------------------------------------------------------------------ elements & operators

template <int N>
struct FElem {  // filtering element
  double A[N * N], b[N], C[N * N], eta[N], J[N * N];
};
template <int N>
struct SElem {  // smoothing element
  double E[N * N], g[N], L[N * N];
};

template <int N>
__host__ __device__ __forceinline__ void f_identity(FElem<N> &e) {
#pragma unroll
  for (int k = 0; k < N * N; ++k) { e.A[k] = (k % (N + 1) == 0) ? 1.0 : 0.0; e.C[k] = 0.0; e.J[k] = 0.0; }
#pragma unroll
  for (int k = 0; k < N; ++k) { e.b[k] = 0.0; e.eta[k] = 0.0; }
}

template <int N>
__host__ __device__ __forceinline__ void f_state(FElem<N> &e, const double *m, const double *C) {
#pragma unroll
  for (int k = 0; k < N * N; ++k) { e.A[k] = 0.0; e.C[k] = C[k]; e.J[k] = 0.0; }
#pragma unroll
  for (int k = 0; k < N; ++k) { e.b[k] = m[k]; e.eta[k] = 0.0; }
}

// inverse of a small matrix for the combine operator (scan only: its contract is 1e-9, so the
// closed forms for n <= 2 need not match dgesv's rounding)
template <int N>
__host__ __device__ __forceinline__ int small_inverse(const double (&Mx)[N * N], double (&inv)[N * N]) {
  if (N == 1) {
    inv[0] = 1.0 / Mx[0];
    return Mx[0] == 0.0 ? BDLM_ST_SINGULAR : 0;
  } else if (N == 2) {
    const double det = Mx[0] * Mx[3] - Mx[2] * Mx[1];
    const double r = 1.0 / det;
    inv[0] = Mx[3] * r; inv[1] = -Mx[1] * r; inv[2] = -Mx[2] * r; inv[3] = Mx[0] * r;
    return det == 0.0 ? BDLM_ST_SINGULAR : 0;
  } else {
    double Mc[N * N];
#pragma unroll
    for (int k = 0; k < N * N; ++k) { Mc[k] = Mx[k]; inv[k] = (k % (N + 1) == 0) ? 1.0 : 0.0; }
    return lu_solve<N, N>(Mc, inv);
  }
}

// out = ei (x) ej, ei earlier in time.  (Appendix C)
// With C_i, J_j symmetric, (I + J_j C_i) = (I + C_i J_j)^T: ONE inverse serves both factors,
//   X = A_j (I + C_i J_j)^-1,   Y = A_i^T (I + J_j C_i)^-1 = ((I + C_i J_j)^-1 A_i)^T.
template <int N>
__host__ __device__ __forceinline__ void f_combine(const FElem<N> &ei, const FElem<N> &ej,
                                                   FElem<N> &out) {
  double Mx[N * N], Minv[N * N], X[N * N], Y[N * N], t1[N * N], t2[N * N], v1[N], v2[N];
  smm<N, N, N, false, false>(ei.C, ej.J, Mx);
#pragma unroll
  for (int k = 0; k < N; ++k) Mx[k * (N + 1)] = 1.0 + Mx[k * (N + 1)];
  small_inverse<N>(Mx, Minv);
  smm<N, N, N, true, true>(Minv, ej.A, X);    // X := M^-T A_j^T = (A_j M^-1)^T
  smm<N, N, N, false, false>(Minv, ei.A, Y);  // Y := M^-1 A_i = (A_i^T M^-T)^T
  // A = (A_j M) A_i
  smm<N, N, N, true, false>(X, ei.A, out.A);
  // b = (A_j M)(b_i + C_i eta_j) + b_j
  smm<N, N, 1, false, false>(ei.C, ej.eta, v1);
#pragma unroll
  for (int k = 0; k < N; ++k) v1[k] = ei.b[k] + v1[k];
  smm<N, N, 1, true, false>(X, v1, v2);
#pragma unroll
  for (int k = 0; k < N; ++k) out.b[k] = v2[k] + ej.b[k];
  // C = (A_j M) C_i A_j^T + C_j
  smm<N, N, N, true, false>(X, ei.C, t1);
  smm<N, N, N, false, true>(t1, ej.A, t2);
#pragma unroll
  for (int k = 0; k < N * N; ++k) out.C[k] = t2[k] + ej.C[k];
  // eta = (A_i^T N)(eta_j - J_j b_i) + eta_i
  smm<N, N, 1, false, false>(ej.J, ei.b, v1);
#pragma unroll
  for (int k = 0; k < N; ++k) v1[k] = ej.eta[k] - v1[k];
  smm<N, N, 1, true, false>(Y, v1, v2);
#pragma unroll
  for (int k = 0; k < N; ++k) out.eta[k] = v2[k] + ei.eta[k];
  // J = (A_i^T N) J_j A_i + J_i
  smm<N, N, N, true, false>(Y, ej.J, t1);
  smm<N, N, N, false, false>(t1, ei.A, t2);
#pragma unroll
  for (int k = 0; k < N * N; ++k) out.J[k] = t2[k] + ei.J[k];
}

// Filtering element of one observation (p = 1): Q = W dt.
template <int N>
__host__ __device__ __forceinline__ void f_element(const double *G, const double *F,
                                                   const double (&Q)[N * N], double V, double y,
                                                   FElem<N> &e) {
  if (isnan(y)) {  // missing: pure prediction
#pragma unroll
    for (int k = 0; k < N * N; ++k) { e.A[k] = G[k]; e.C[k] = Q[k]; e.J[k] = 0.0; }
#pragma unroll
    for (int k = 0; k < N; ++k) { e.b[k] = 0.0; e.eta[k] = 0.0; }
    return;
  }
  double QF[N], GtF[N], K[N], IKH[N * N], S;
  smm<N, N, 1, false, false>(Q, F, QF);
  smm<1, N, 1, true, false>(F, QF, &S);
  S = S + V;
  smm<N, N, 1, true, false>(G, F, GtF);  // G^T F
#pragma unroll
  for (int i = 0; i < N; ++i) K[i] = QF[i] / S;
#pragma unroll
  for (int j = 0; j < N; ++j)
#pragma unroll
    for (int i = 0; i < N; ++i) IKH[i + j * N] = ((i == j) ? 1.0 : 0.0) - K[i] * F[j];
  smm<N, N, N, false, false>(IKH, G, e.A);
  smm<N, N, N, false, false>(IKH, Q, e.C);
#pragma unroll
  for (int i = 0; i < N; ++i) { e.b[i] = K[i] * y; e.eta[i] = GtF[i] * y / S; }
#pragma unroll
  for (int j = 0; j < N; ++j)
#pragma unroll
    for (int i = 0; i < N; ++i) e.J[i + j * N] = GtF[i] * GtF[j] / S;
}

template <int N>
__host__ __device__ __forceinline__ void s_identity(SElem<N> &e) {
#pragma unroll
  for (int k = 0; k < N * N; ++k) { e.E[k] = (k % (N + 1) == 0) ? 1.0 : 0.0; e.L[k] = 0.0; }
#pragma unroll
  for (int k = 0; k < N; ++k) e.g[k] = 0.0;
}

template <int N>
__host__ __device__ __forceinline__ void s_state(SElem<N> &e, const double *s, const double *S) {
#pragma unroll
  for (int k = 0; k < N * N; ++k) { e.E[k] = 0.0; e.L[k] = S[k]; }
#pragma unroll
  for (int k = 0; k < N; ++k) e.g[k] = s[k];
}

// out = ei (x) ej, ei earlier:  E = E_i E_j ; g = E_i g_j + g_i ; L = E_i L_j E_i^T + L_i
template <int N>
__host__ __device__ __forceinline__ void s_combine(const SElem<N> &ei, const SElem<N> &ej,
                                                   SElem<N> &out) {
  double t1[N * N], t2[N * N], v[N];
  smm<N, N, N, false, false>(ei.E, ej.E, out.E);
  smm<N, N, 1, false, false>(ei.E, ej.g, v);
#pragma unroll
  for (int k = 0; k < N; ++k) out.g[k] = v[k] + ei.g[k];
  smm<N, N, N, false, false>(ei.E, ej.L, t1);
  smm<N, N, N, false, true>(t1, ei.E, t2);
#pragma unroll
  for (int k = 0; k < N * N; ++k) out.L[k] = t2[k] + ei.L[k];
}

// Smoothing element of a filtered row that has a successor: E = C G^T R1^-1 (the RTS gain),
// g = m - E a1, L = C - E R1 E^T, with (a1, R1) the one-step prediction from (m, C).
template <int N>
__host__ __device__ __forceinline__ void s_element_pred(const double *G, const double (&m)[N],
                                                        const double (&C)[N * N], const double (&a1)[N],
                                                        const double (&R1)[N * N], SElem<N> &e) {
  double CGt[N * N], Rinv[N * N], t1[N * N], t2[N * N], v[N];
  smm<N, N, N, false, true>(C, G, CGt);
  small_inverse<N>(R1, Rinv);
  smm<N, N, N, false, false>(CGt, Rinv, e.E);  // E = C G^T R1^-1
  smm<N, N, 1, false, false>(e.E, a1, v);
#pragma unroll
  for (int k = 0; k < N; ++k) e.g[k] = m[k] - v[k];
  smm<N, N, N, false, false>(e.E, R1, t1);
  smm<N, N, N, false, true>(t1, e.E, t2);
#pragma unroll
  for (int k = 0; k < N * N; ++k) e.L[k] = C[k] - t2[k];
}

namespace {

// Most ROWS per thread (level 1; a multiple of kGrp); scan_rows_per_thread picks at most this many
// per call.  64 beat 32 and 16, and 128 gained nothing (profiles/r2_tuning.txt, "scan level-1
// granularity" and "kSub = 128").
constexpr int kSub = 64;
constexpr int kGrp = 4;        // rows per vector group: 4 rows x K doubles = K 32-byte sectors
constexpr int kScanBlock = 256;
constexpr size_t kScanTableBytes = (size_t)64 << 10;

template <int N>
struct ScanModel {
  double G[N * N], F[N], W[N * N], V;
};

// Thread c owns OUTPUT ROWS [c*kSub, (c+1)*kSub) (row = t + keep_init), so that every group of
// kGrp rows of every output field is a run of whole, 32-byte-aligned sectors that the owning
// thread alone writes with 256-bit stores.  With one thread per 64 consecutive rows a store
// instruction can never be coalesced ACROSS threads; what matters is that no sector is written
// piecemeal: the partially written lines of all resident threads (6 fields x 128 B x 2.6e5
// threads at T = 2^24) exceed L2, so 8-byte stores were evicted half-filled and cost a DRAM
// read-fill plus a second write (ncu: 245 MB read, 596 MB written for 470 MB of output).
__device__ __forceinline__ int64_t first_step(int64_t c, int keep_init, int sub) {
  const int64_t t = c * (int64_t)sub - keep_init;
  return t < 0 ? 0 : t;
}

__device__ __forceinline__ void st_v4(double *p, double a, double b, double c, double d) {
  asm volatile("st.global.cs.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d)
               : "memory");
}
__device__ __forceinline__ void ld_v4(const double *p, double *x) {
  asm volatile("ld.global.v4.f64 {%0, %1, %2, %3}, [%4];"
               : "=d"(x[0]), "=d"(x[1]), "=d"(x[2]), "=d"(x[3]) : "l"(p));
}
__device__ __forceinline__ void ld_v2(const double *p, double *x) {
  asm volatile("ld.global.v2.f64 {%0, %1}, [%2];" : "=d"(x[0]), "=d"(x[1]) : "l"(p));
}

// One row of a dense field (K contiguous doubles), widest aligned loads available.
template <int K, bool VEC>
__device__ __forceinline__ void load_row(const View &v, int64_t row, double (&x)[K]) {
  const double *p = v.ptr + row * v.sr;
  if (VEC && K % 4 == 0) {
#pragma unroll
    for (int k = 0; k < K; k += 4) ld_v4(p + k, x + k);
  } else if (VEC && K % 2 == 0) {
#pragma unroll
    for (int k = 0; k < K; k += 2) ld_v2(p + k, x + k);
  } else {
#pragma unroll
    for (int k = 0; k < K; ++k) x[k] = ld_stream(p + k * v.sk);
  }
}

// Observations behind a group of kGrp rows [r, r + kGrp): y[r - keep_init + i].  Thread-private
// streams must be fetched a whole aligned 32-byte sector (better: line) at a time -- 8-byte loads
// spread over four steps were re-fetched from DRAM up to 4x (the sector is evicted between the
// steps; ncu: 675 MB read for 168 MB of input).  With keep_init the rows are one observation
// ahead of the aligned sector, so the last element of each sector is carried to the next group.
template <bool VEC>
struct YGroup {
  double carry;
  __device__ __forceinline__ void start(const double *y, int64_t r0, int keep_init) {
    carry = (VEC && keep_init && r0 > 0) ? y[r0 - 1] : 0.0;
  }
  // precondition: rows r .. r + kGrp - 1 all exist (r + kGrp <= T + keep_init)
  __device__ __forceinline__ void load(const double *y, int64_t r, int64_t T, int keep_init,
                                       double (&yv)[kGrp]) {
    if (VEC) {
      double v[kGrp];
      if (r + kGrp <= T) ld_v4(y + r, v);
      else {
#pragma unroll
        for (int i = 0; i < kGrp; ++i) v[i] = (r + i < T) ? y[r + i] : 0.0;
      }
      if (keep_init) {
        yv[0] = carry;
#pragma unroll
        for (int i = 1; i < kGrp; ++i) yv[i] = v[i - 1];
        carry = v[kGrp - 1];
      } else {
#pragma unroll
        for (int i = 0; i < kGrp; ++i) yv[i] = v[i];
      }
    } else {
#pragma unroll
      for (int i = 0; i < kGrp; ++i) {
        const int64_t t = r + i - keep_init;
        yv[i] = t >= 0 ? y[t] : 0.0;
      }
    }
  }
};

// Per-step observation vectors behind a group of kGrp rows (f_tv): F[t] = F + t*N, t = r - keep_init + i,
// fetched like YGroup fetches y -- the N sectors of steps r .. r + kGrp - 1 at once, the last step's
// vector carried to the next group when keep_init puts the rows one step ahead of the sectors.
template <int N, bool VEC>
struct FGroup {
  double carry[N];
  __device__ __forceinline__ void start(const double *F, int64_t r0, int keep_init) {
#pragma unroll
    for (int k = 0; k < N; ++k) carry[k] = (VEC && keep_init && r0 > 0) ? F[(r0 - 1) * N + k] : 0.0;
  }
  // precondition as YGroup::load; a row before the first step (the prior) gets zeros
  __device__ __forceinline__ void load(const double *F, int64_t r, int64_t T, int keep_init,
                                       double (&fv)[kGrp][N]) {
    if (VEC) {
      double v[kGrp * N];
      if (r + kGrp <= T) {
#pragma unroll
        for (int k = 0; k < kGrp * N; k += 4) ld_v4(F + r * N + k, v + k);
      } else {
#pragma unroll
        for (int k = 0; k < kGrp * N; ++k) v[k] = (r + k / N < T) ? F[r * N + k] : 0.0;
      }
#pragma unroll
      for (int i = 0; i < kGrp; ++i)
#pragma unroll
        for (int k = 0; k < N; ++k) {
          if (keep_init) fv[i][k] = i == 0 ? carry[k] : v[(i - 1) * N + k];
          else fv[i][k] = v[i * N + k];
        }
      if (keep_init) {
#pragma unroll
        for (int k = 0; k < N; ++k) carry[k] = v[(kGrp - 1) * N + k];
      }
    } else {
#pragma unroll
      for (int i = 0; i < kGrp; ++i) {
        const int64_t t = r + i - keep_init;
#pragma unroll
        for (int k = 0; k < N; ++k) fv[i][k] = t >= 0 ? F[t * N + k] : 0.0;
      }
    }
  }
};

// kGrp consecutive rows of a dense field in one go (whole lines for K >= 4).
template <int K>
__device__ __forceinline__ void load_group(const View &v, int64_t row, double (&x)[kGrp * K]) {
  const double *p = v.ptr + row * K;
#pragma unroll
  for (int k = 0; k < kGrp * K; k += 4) ld_v4(p + k, x + k);
}

// Group buffer of one field: kGrp rows x K doubles in registers (all indices are compile-time
// after unrolling, so only the not-yet-flushed tail stays live).  put<I>() deposits row I of
// the group and flushes every 32-byte chunk that has just become complete; ASC = rows arrive in
// increasing order (filter), otherwise decreasing (smoother).
template <int K>
struct GroupBuf {
  double g[kGrp * K];
  template <int I, bool ASC>
  __device__ __forceinline__ void put(double *base, const double *x) {
#pragma unroll
    for (int k = 0; k < K; ++k) g[I * K + k] = x[k];
    constexpr int lo = ASC ? (I * K / 4) * 4 : ((I * K + 3) / 4) * 4;
    constexpr int hi = ASC ? ((I + 1) * K / 4) * 4 : (((I + 1) * K + 3) / 4) * 4;
#pragma unroll
    for (int q = lo; q < hi && q < kGrp * K; q += 4) st_v4(base + q, g[q], g[q + 1], g[q + 2], g[q + 3]);
  }
};

template <int K>
__device__ __forceinline__ void store_row_scalar(const View &v, int64_t row, const double *x) {
  if (!v.ptr) return;
  double *p = v.ptr + row * v.sr;
#pragma unroll
  for (int k = 0; k < K; ++k) st_stream(p + k * v.sk, x[k]);
}

// ---- level 1, forward: per-thread aggregate over the observations behind its rows.
//
// Time-invariant model, regular grid, no missing value in the thread's range (the common case):
// the element of an observed step is (A1, K y, C1, h y, J1) with y-independent A1, C1, J1, K, h,
// so the (A, C, J) parts of the k-step aggregate acc_k = e(y_0) (x) ... (x) e(y_{k-1}) are the same
// for every thread and only (b, eta) depend on the data -- linearly:
//     b_{k+1}   = X_k b_k + u_k y_k            X_k = A1 (I + C_k J1)^-1,  u_k = X_k C_k h + K
//     eta_{k+1} = eta_k + v_k y_k - Z_k b_k    Y_k = A_k^T (I + J1 C_k)^-1,  v_k = Y_k h,  Z_k = Y_k J1
// The host composes acc_1..acc_kSub once (kSub generic combines) and uploads the table; a thread
// then spends 2N^2 + 2N multiply-adds per step instead of a generic combine (two LU solves and
// ten small products).  A thread that meets a NaN recomputes its range generically.
template <int N>
struct FwdTable {
  struct Step { double X[N * N], u[N], v[N], Z[N * N]; } step[kSub];  // step[k]: acc_k -> acc_{k+1}
  struct Agg { double A[N * N], C[N * N], J[N * N]; } agg[kSub + 1];  // agg[k]: parts of acc_k
  double K[N], h[N];
};

template <int N>
void build_fwd_table(const ScanModel<N> &md, FwdTable<N> &tb) {
  FElem<N> e1, acc, nxt;
  f_element<N>(md.G, md.F, md.W, md.V, 1.0, e1);  // y = 1: b = K, eta = h
  for (int i = 0; i < N; ++i) { tb.K[i] = e1.b[i]; tb.h[i] = e1.eta[i]; }
  acc = e1;
  for (int k = 1; k <= kSub; ++k) {
    for (int q = 0; q < N * N; ++q) { tb.agg[k].A[q] = acc.A[q]; tb.agg[k].C[q] = acc.C[q]; tb.agg[k].J[q] = acc.J[q]; }
    if (k == kSub) break;
    // X_k, Y_k exactly as f_combine forms them
    double CJ[N * N], Mt[N * N], X[N * N], JC[N * N], Nt[N * N], Y[N * N], Xm[N * N], Ym[N * N], t[N];
    smm<N, N, N, false, false>(acc.C, e1.J, CJ);
    smm<N, N, N, false, false>(e1.J, acc.C, JC);
    for (int j = 0; j < N; ++j)
      for (int i = 0; i < N; ++i) {
        Mt[i + j * N] = ((i == j) ? 1.0 : 0.0) + CJ[j + i * N];
        X[i + j * N] = e1.A[j + i * N];
        Nt[i + j * N] = ((i == j) ? 1.0 : 0.0) + JC[j + i * N];
        Y[i + j * N] = acc.A[i + j * N];
      }
    lu_solve<N, N>(Mt, X);  // X = (A1 M)^T
    lu_solve<N, N>(Nt, Y);  // Y = (A_k^T N)^T
    for (int j = 0; j < N; ++j)
      for (int i = 0; i < N; ++i) { Xm[i + j * N] = X[j + i * N]; Ym[i + j * N] = Y[j + i * N]; }
    typename FwdTable<N>::Step &sp = tb.step[k];
    for (int q = 0; q < N * N; ++q) sp.X[q] = Xm[q];
    smm<N, N, 1, false, false>(acc.C, tb.h, t);
    smm<N, N, 1, false, false>(Xm, t, sp.u);
    for (int i = 0; i < N; ++i) sp.u[i] = sp.u[i] + tb.K[i];
    smm<N, N, 1, false, false>(Ym, tb.h, sp.v);
    smm<N, N, N, false, false>(Ym, e1.J, sp.Z);
    f_combine<N>(acc, e1, nxt);
    acc = nxt;
  }
}

// (m, C) or (s, S) handed over by value: no host buffer outlives the call.
template <int N>
struct StateArg {
  double v[N + N * N];
};
template <int N>
StateArg<N> state_arg(const double *host) {
  StateArg<N> s;
  for (int k = 0; k < N + N * N; ++k) s.v[k] = host ? host[k] : 0.0;
  return s;
}

//
// FTV (f_tv, per-step F[t] = Fd + t*N): no table -- the steps' (A, C, J) differ -- so every thread
// composes its steps with the generic combine, reading F like y.
template <int N, bool VEC, bool FTV = false>
__global__ void __launch_bounds__(128)
fwd_reduce_kernel(const ScanModel<N> md, const FwdTable<N> *__restrict__ tb,
                  const double *__restrict__ y, int64_t T, int64_t M, int keep_init,
                  FElem<N> *agg /* [M + 1], slot 0 = the start element */,
                  const StateArg<N> start, bool identity_start, int sub,
                  const double *__restrict__ Fd /* FTV: [T][N] */) {
  const int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (c >= M) return;
  if (c == 0) {  // slot 0: the state before the chunk, or the identity (aggregate-only phases)
    FElem<N> e0;
    if (identity_start) f_identity<N>(e0); else f_state<N>(e0, start.v, start.v + N);
    agg[0] = e0;
  }
  const int64_t rows = T + keep_init;
  const int64_t r0 = c * (int64_t)sub, r1 = (r0 + sub < rows) ? r0 + sub : rows;
  if constexpr (FTV) {
    FElem<N> acc, e, tmp;
    bool have = false;
    auto fold = [&](const double *Ft, double yt) {
      f_element<N>(md.G, Ft, md.W, md.V, yt, e);
      if (have) { f_combine<N>(acc, e, tmp); acc = tmp; }
      else { acc = e; have = true; }
    };
    YGroup<VEC> yg;
    FGroup<N, VEC> fg;
    yg.start(y, r0, keep_init);
    fg.start(Fd, r0, keep_init);
    int64_t r = r0;
    for (; r + kGrp <= r1; r += kGrp) {
      double yv[kGrp], fv[kGrp][N];
      yg.load(y, r, T, keep_init, yv);
      fg.load(Fd, r, T, keep_init, fv);
#pragma unroll
      for (int i = 0; i < kGrp; ++i)
        if (r + i >= keep_init) fold(fv[i], yv[i]);
    }
    for (; r < r1; ++r)
      if (r >= keep_init) fold(Fd + (r - keep_init) * N, y[r - keep_init]);
    agg[c + 1] = acc;
    return;
  }
  const int64_t t0 = first_step(c, keep_init, sub), t1 = r1 - keep_init;
  double b[N], eta[N];
#pragma unroll
  for (int i = 0; i < N; ++i) { b[i] = 0.0; eta[i] = 0.0; }
  bool missing = false;
  int k = 0;  // steps composed so far
  auto step = [&](double yk) {
    missing |= isnan(yk);
    if (k == 0) {
#pragma unroll
      for (int i = 0; i < N; ++i) { b[i] = tb->K[i] * yk; eta[i] = tb->h[i] * yk; }
    } else {
      const typename FwdTable<N>::Step &sp = tb->step[k];
      double nb[N], ne[N];
#pragma unroll
      for (int i = 0; i < N; ++i) {
        double xb = 0.0, zb = 0.0;
#pragma unroll
        for (int j = 0; j < N; ++j) { xb += sp.X[i + j * N] * b[j]; zb += sp.Z[i + j * N] * b[j]; }
        nb[i] = xb + sp.u[i] * yk;
        ne[i] = eta[i] + sp.v[i] * yk - zb;
      }
#pragma unroll
      for (int i = 0; i < N; ++i) { b[i] = nb[i]; eta[i] = ne[i]; }
    }
    ++k;
  };
  YGroup<VEC> yg;
  yg.start(y, r0, keep_init);
  int64_t r = r0;
  for (; r + kGrp <= r1; r += kGrp) {
    double yv[kGrp];
    yg.load(y, r, T, keep_init, yv);
#pragma unroll
    for (int i = 0; i < kGrp; ++i)
      if (r + i >= keep_init) step(yv[i]);  // row 0 of a keep_init run is the prior, not a step
  }
  for (; r < r1; ++r)
    if (r >= keep_init) step(y[r - keep_init]);
  if (!missing) {
    FElem<N> &o = agg[c + 1];
#pragma unroll
    for (int q = 0; q < N * N; ++q) { o.A[q] = tb->agg[k].A[q]; o.C[q] = tb->agg[k].C[q]; o.J[q] = tb->agg[k].J[q]; }
#pragma unroll
    for (int i = 0; i < N; ++i) { o.b[i] = b[i]; o.eta[i] = eta[i]; }
    return;
  }
  // generic path: a missing observation changes the element's (A, C, J)
  FElem<N> acc, e, tmp;
  f_element<N>(md.G, md.F, md.W, md.V, y[t0], acc);
  for (int64_t t = t0 + 1; t < t1; ++t) {
    f_element<N>(md.G, md.F, md.W, md.V, y[t], e);
    f_combine<N>(acc, e, tmp);
    acc = tmp;
  }
  agg[c + 1] = acc;
}

// ---- level 2: inclusive scan of an element array with an associative operator.
// IDXREV: scan position p maps to array index M-1-p (suffix scan).  OPREV: an element later
// in SCAN order is EARLIER in time (so it is the left operand).  The top level of a suffix
// scan uses (IDXREV, OPREV) = (true, true); its block totals are stored in scan order and
// are therefore scanned with (false, true).
template <class E>
struct Op;
template <int N>
struct Op<FElem<N>> {
  __device__ static void apply(const FElem<N> &earlier, const FElem<N> &later, FElem<N> &o) {
    f_combine<N>(earlier, later, o);
  }
};
template <int N>
struct Op<SElem<N>> {
  __device__ static void apply(const SElem<N> &earlier, const SElem<N> &later, SElem<N> &o) {
    s_combine<N>(earlier, later, o);
  }
};

// first (x) second in SCAN order
template <class E, bool OPREV>
__device__ __forceinline__ void scan_comb(const E &first, const E &second, E &o) {
  if (OPREV) Op<E>::apply(second, first, o);
  else Op<E>::apply(first, second, o);
}

// A block scans kScanBlock * kPer consecutive positions: every thread folds its kPer elements
// serially (kPer - 1 combines), the thread totals go through a Hillis-Steele scan in shared
// memory (log2(kScanBlock) combines per THREAD, i.e. 2 per element), and a second serial sweep
// applies the exclusive prefix (kPer combines).  3.75 combines per element instead of 8 -- the
// combine (two LU solves + ten products) is what this level costs.
constexpr int kPer = 4;

// Shared-memory staging of the thread totals is component-major ([k][thread]): an element is 10-56
// doubles, so element-major rows would put every lane of a warp on the same banks.
template <class E>
__device__ __forceinline__ void sm_put(double *buf, int i, const E &e) {
  constexpr int kD = (int)(sizeof(E) / sizeof(double));
  const double *s = reinterpret_cast<const double *>(&e);
#pragma unroll
  for (int k = 0; k < kD; ++k) buf[k * kScanBlock + i] = s[k];
}
template <class E>
__device__ __forceinline__ void sm_get(const double *buf, int i, E &e) {
  constexpr int kD = (int)(sizeof(E) / sizeof(double));
  double *d = reinterpret_cast<double *>(&e);
#pragma unroll
  for (int k = 0; k < kD; ++k) d[k] = buf[k * kScanBlock + i];
}

template <class E, bool IDXREV, bool OPREV>
__global__ void __launch_bounds__(kScanBlock)
block_scan_kernel(E *x, int64_t M, E *totals) {
  extern __shared__ unsigned char raw[];
  constexpr int kD = (int)(sizeof(E) / sizeof(double));
  double *buf0 = reinterpret_cast<double *>(raw), *buf1 = buf0 + kD * kScanBlock;
  const int tid = threadIdx.x;
  const int64_t base = (int64_t)blockIdx.x * (kScanBlock * kPer);
  const int64_t p0 = base + (int64_t)tid * kPer;
  const int cnt = (p0 >= M) ? 0 : (int)((M - p0 < kPer) ? (M - p0) : kPer);
  auto at = [&](int64_t p) -> E & { return x[IDXREV ? (M - 1 - p) : p]; };
  const bool act = cnt > 0;
  E mine;  // this thread's running total (scan order)
  if (act) {
    E o;
    mine = at(p0);
    for (int j = 1; j < cnt; ++j) { scan_comb<E, OPREV>(mine, at(p0 + j), o); mine = o; }
    sm_put<E>(buf0, tid, mine);
  }
  __syncthreads();
  double *src = buf0, *dst = buf1;
  for (int off = 1; off < kScanBlock; off <<= 1) {
    if (act) {
      if (tid >= off) {
        E prev, o;
        sm_get<E>(src, tid - off, prev);
        scan_comb<E, OPREV>(prev, mine, o);
        mine = o;
      }
      sm_put<E>(dst, tid, mine);
    }
    __syncthreads();
    double *t = src; src = dst; dst = t;
  }
  if (act) {
    E run, o;
    if (tid > 0) {
      E prev;
      sm_get<E>(src, tid - 1, prev);
      scan_comb<E, OPREV>(prev, at(p0), o); run = o; at(p0) = run;
    } else {
      run = at(p0);
    }
    for (int j = 1; j < cnt; ++j) { scan_comb<E, OPREV>(run, at(p0 + j), o); run = o; at(p0 + j) = run; }
  }
  const int64_t left = M - base;  // positions in this block
  const int last = (int)(((left < kScanBlock * kPer ? left : kScanBlock * kPer) - 1) / kPer);
  if (totals && tid == last) totals[blockIdx.x] = mine;
}

template <class E, bool IDXREV, bool OPREV>
__global__ void __launch_bounds__(kScanBlock)
add_prefix_kernel(E *x, int64_t M, const E *totals /* scanned, scan order */) {
  if (blockIdx.x == 0) return;
  const E pre = totals[blockIdx.x - 1];
#pragma unroll 1
  for (int j = 0; j < kPer; ++j) {
    const int64_t p = (int64_t)blockIdx.x * (kScanBlock * kPer) + j * kScanBlock + threadIdx.x;
    if (p >= M) return;
    const int64_t idx = IDXREV ? (M - 1 - p) : p;
    const E cur = x[idx];
    E o;
    scan_comb<E, OPREV>(pre, cur, o);
    x[idx] = o;
  }
}

// defer_top: leave the top level's block prefixes unapplied -- the consumer (apply sweep) composes
// scratch[block - 1] itself, which saves a read-modify-write pass over the whole element array.
template <class E, bool IDXREV, bool OPREV>
cudaError_t device_scan(E *x, int64_t M, E *scratch, cudaStream_t stream, int64_t *launches,
                        bool defer_top = false) {
  if (M <= 1) return cudaSuccess;
  const int64_t per_block = kScanBlock * kPer;
  const int64_t nb = (M + per_block - 1) / per_block;
  const size_t smem = 2 * kScanBlock * sizeof(E);
  cudaError_t e = cudaFuncSetAttribute(block_scan_kernel<E, IDXREV, OPREV>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  block_scan_kernel<E, IDXREV, OPREV><<<(unsigned)nb, kScanBlock, smem, stream>>>(
      x, M, nb > 1 ? scratch : nullptr);
  ++*launches;
  if (nb > 1) {
    e = device_scan<E, false, OPREV>(scratch, nb, scratch + nb, stream, launches);
    if (e != cudaSuccess) return e;
    if (!defer_top) {
      add_prefix_kernel<E, IDXREV, OPREV><<<(unsigned)nb, kScanBlock, 0, stream>>>(x, M, scratch);
      ++*launches;
    }
  }
  return cudaGetLastError();
}

// ---- apply, forward: sequential Kalman recursion from the scanned start state
template <int N>
struct FwdRow {  // everything KfState holds for one row
  double a[N], R[N * N], f, Q, m[N], C[N * N];
};

// One output row.  (an, Rn) is the prediction INTO this row, carried from the previous row
// (it doubles as the (a1, R1) of the previous row's smoothing element); on return it is the
// prediction into the next row.  FUSE: also fold this row's smoothing element into sacc when the
// row has a successor (r < nrows), which saves the smoother's level-1 pass over (m, C).
template <int N, bool FUSE>
__device__ __forceinline__ void fwd_row(const ScanModel<N> &md, const double *F /* this row's */,
                                        const double (&W)[N * N], bool init_row,
                                        double yv, double (&m)[N], double (&C)[N * N],
                                        double (&an)[N], double (&Rn)[N * N], FwdRow<N> &o, int &st,
                                        bool has_succ, SElem<N> &sacc, bool &shave) {
  if (init_row) {  // KalmanFilter.initialiseState: a = m = m0, R = C = C0, f, Q = None
    const double nanv = __longlong_as_double(0x7ff8000000000000LL);
#pragma unroll
    for (int k = 0; k < N; ++k) o.a[k] = m[k];
#pragma unroll
    for (int k = 0; k < N * N; ++k) o.R[k] = C[k];
    o.f = nanv; o.Q = nanv;
  } else {
#pragma unroll
    for (int k = 0; k < N; ++k) o.a[k] = an[k];
#pragma unroll
    for (int k = 0; k < N * N; ++k) o.R[k] = Rn[k];
    update<N, true>(F, md.V, yv, o.a, o.R, o.f, o.Q, m, C, st);
  }
#pragma unroll
  for (int k = 0; k < N; ++k) o.m[k] = m[k];
#pragma unroll
  for (int k = 0; k < N * N; ++k) o.C[k] = C[k];
  advance<N, true>(md.G, W, 1.0, m, C, an, Rn);
  if (FUSE && has_succ) {
    SElem<N> e, tmp;
    s_element_pred<N>(md.G, m, C, an, Rn, e);
    if (shave) { s_combine<N>(sacc, e, tmp); sacc = tmp; }
    else { sacc = e; shave = true; }
  }
}

// Filtered (m, C) of the row before thread c's first row on one GPU: (b, C) of its exclusive prefix
// pre[c], composed with the top-level block prefix that device_scan left unapplied (defer_top).
// fwd_apply_kernel inlines the same composition (plus the multi-GPU carry) by hand: calling this
// function from it reorders its SASS.
template <int N>
__device__ __forceinline__ void fwd_start_state(const FElem<N> *pre, int64_t c, const FElem<N> *tot,
                                                double (&m)[N], double (&C)[N * N]) {
  const int64_t blk = c / (kScanBlock * kPer);  // level-2 block of scan position c
  if (tot && blk > 0) {
    FElem<N> o;  // only (b, C) is live, the rest folds away
    f_combine<N>(tot[blk - 1], pre[c], o);
#pragma unroll
    for (int k = 0; k < N; ++k) m[k] = o.b[k];
#pragma unroll
    for (int k = 0; k < N * N; ++k) C[k] = o.C[k];
  } else {
#pragma unroll
    for (int k = 0; k < N; ++k) m[k] = pre[c].b[k];
#pragma unroll
    for (int k = 0; k < N * N; ++k) C[k] = pre[c].C[k];
  }
}

// The two apply sweeps ask ptxas for one resident block per SM: asking for more makes them spill,
// which costs more than the occupancy gains (profiles/r1_tuning.txt, "scan apply sweeps").
// FTV: row r updates with F[t] = Fd + t*N, t = r - keep_init.
template <int N, bool VEC, bool FUSE, bool FTV = false>
__global__ void __launch_bounds__(128, 1)
fwd_apply_kernel(const ScanModel<N> md, const double *__restrict__ y, int64_t T, int64_t M,
                 const FElem<N> *pre /* [M+1] inclusive scan with slot 0 = start */,
                 int keep_init, KfViews kf, int32_t *status,
                 SElem<N> *sagg /* FUSE: smoother level-1 aggregates */, int64_t nrows,
                 const FElem<N> *carry /* multi-GPU: everything before this chunk, or nullptr */,
                 const FElem<N> *tot /* scanned level-2 block totals whose prefix `pre` still lacks, or nullptr */,
                 int sub, const double *__restrict__ Fd /* FTV: [T][N] */) {
  const int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (c >= M) return;
  const int64_t rows = T + keep_init;
  const int64_t r0 = c * (int64_t)sub, r1 = (r0 + sub < rows) ? r0 + sub : rows;
  double m[N], C[N * N], W[N * N], an[N], Rn[N * N];
  int st = 0;
  const int64_t blk = c / (kScanBlock * kPer);  // level-2 block of scan position c
  const bool use_tot = tot && blk > 0;
  if (carry || use_tot) {
    // the scan ran with an identity start (carry) and / or left its top-level block prefix to us:
    // compose them on the fly; only (b, C) of the result is live, the rest folds away
    FElem<N> left, o;
    if (carry && use_tot) f_combine<N>(*carry, tot[blk - 1], left);
    else left = carry ? *carry : tot[blk - 1];
    f_combine<N>(left, pre[c], o);
#pragma unroll
    for (int k = 0; k < N; ++k) m[k] = o.b[k];
#pragma unroll
    for (int k = 0; k < N * N; ++k) C[k] = o.C[k];
  } else {
#pragma unroll
    for (int k = 0; k < N; ++k) m[k] = pre[c].b[k];
#pragma unroll
    for (int k = 0; k < N * N; ++k) C[k] = pre[c].C[k];
  }
#pragma unroll
  for (int k = 0; k < N * N; ++k) W[k] = md.W[k];
  advance<N, true>(md.G, W, 1.0, m, C, an, Rn);
  SElem<N> sacc;
  bool shave = false;
  int64_t r = r0;
  if (VEC) {
    YGroup<true> yg;
    FGroup<N, true> fg;
    yg.start(y, r0, keep_init);
    if constexpr (FTV) fg.start(Fd, r0, keep_init);
    for (; r + kGrp <= r1; r += kGrp) {
      double yv[kGrp], fv[kGrp][N];
      yg.load(y, r, T, keep_init, yv);
      if constexpr (FTV) fg.load(Fd, r, T, keep_init, fv);
      GroupBuf<N> ga, gm;
      GroupBuf<N * N> gR, gC;
      GroupBuf<1> gf, gQ;
#define BDLM_FWD_ROW(I)                                                          \
  {                                                                              \
    FwdRow<N> o;                                                                 \
    fwd_row<N, FUSE>(md, FTV ? fv[I] : md.F, W, keep_init && r + I == 0, yv[I],  \
                     m, C, an, Rn, o, st, r + I < nrows, sacc, shave);           \
    if (kf.a.ptr) ga.template put<I, true>(kf.a.ptr + r * N, o.a);               \
    if (kf.R.ptr) gR.template put<I, true>(kf.R.ptr + r * (N * N), o.R);         \
    if (kf.f.ptr) gf.template put<I, true>(kf.f.ptr + r, &o.f);                  \
    if (kf.Q.ptr) gQ.template put<I, true>(kf.Q.ptr + r, &o.Q);                  \
    if (kf.m.ptr) gm.template put<I, true>(kf.m.ptr + r * N, o.m);               \
    if (kf.C.ptr) gC.template put<I, true>(kf.C.ptr + r * (N * N), o.C);         \
  }
      BDLM_FWD_ROW(0) BDLM_FWD_ROW(1) BDLM_FWD_ROW(2) BDLM_FWD_ROW(3)
#undef BDLM_FWD_ROW
    }
  }
  for (; r < r1; ++r) {  // ragged tail (or unaligned / strided outputs): scalar stores
    const int64_t t = r - keep_init;
    FwdRow<N> o;
    fwd_row<N, FUSE>(md, (FTV && t >= 0) ? Fd + t * N : md.F, W, t < 0, t >= 0 ? y[t] : 0.0, m, C, an, Rn, o,
                     st, r < nrows, sacc, shave);
    store_row_scalar<N>(kf.a, r, o.a); store_row_scalar<N * N>(kf.R, r, o.R);
    store_row_scalar<1>(kf.f, r, &o.f); store_row_scalar<1>(kf.Q, r, &o.Q);
    store_row_scalar<N>(kf.m, r, o.m); store_row_scalar<N * N>(kf.C, r, o.C);
  }
  if (FUSE && shave) sagg[c] = sacc;
  if (status && st) atomicOr(status, st);
}

// ---- log-likelihoods + last filtered state (bdlm_scan_loglik): the forward apply recursion of
// one thread's rows with nothing stored per row.  keep_init = 1: row 0 is the prior, row r holds
// step t = r - 1.  Per row (after the update) the thread adds, in row order,
//   TR:          log N(m_t; a_t, W), a_t = G m_{t-1} being the prediction fwd_row carries in;
//   innovations: -dd^2/2 - log(sqrt(2 pi) sd), sd = sqrt(Q_t), dd = (y_t - f_t) / sd, y_t observed
// (scalar_filters.cu loglik_small_kernel's terms).  The block's thread sums then go through a
// fixed-order tree in shared memory to one LoglikPart per block, which loglik_finish_kernel sums in
// a fixed order: no atomics, so a call gives the same bits on any stream or context.
struct LoglikPart {
  double tr, in;
  int st;
};
constexpr int kLlBlock = 128, kLlFinish = 256;

// DIST: one rank's chunk of a time-sharded series (bdlm_scan_dist_loglik_partial).  Its scan ran with
// an identity start, so every thread composes `carry` (the prior and every earlier chunk, i.e. the
// filtered state at the end of the previous chunk) in front of its prefix, as fwd_apply_kernel does;
// keep_init = 0 on every rank but the first, where row r then holds step t = r.
// FTV: row r updates with F[t] = Fd + t*N, as fwd_apply_kernel.
template <int N, bool VEC, bool TR, bool DIST, bool FTV = false>
__global__ void __launch_bounds__(kLlBlock)
fwd_loglik_kernel(const ScanModel<N> md, const double *__restrict__ y, int64_t T, int64_t M,
                  const FElem<N> *pre /* [M+1] inclusive scan with slot 0 = the prior */,
                  const FElem<N> *tot /* scanned level-2 block totals `pre` still lacks, or nullptr */,
                  int sub, LoglikPart *part /* [gridDim.x] */, double *last /* [N + N*N]: (m_T, C_T) */,
                  int keep_init /* DIST */, const FElem<N> *carry /* DIST */,
                  const double *__restrict__ Fd /* FTV: [T][N] */) {
  __shared__ double s_tr[kLlBlock], s_in[kLlBlock];
  __shared__ int s_st[kLlBlock];
  const int tid = threadIdx.x;
  const int64_t c = blockIdx.x * (int64_t)blockDim.x + tid;
  const int ki = DIST ? keep_init : 1;
  double tr = 0.0, li = 0.0;
  int st = 0;
  if (c < M) {
    const int64_t rows = T + ki;
    const int64_t r0 = c * (int64_t)sub, r1 = (r0 + sub < rows) ? r0 + sub : rows;
    double m[N], C[N * N], W[N * N], an[N], Rn[N * N];
    if constexpr (DIST) {
      const int64_t blk = c / (kScanBlock * kPer);
      FElem<N> o;  // only (b, C) is live
      if (tot && blk > 0) {
        FElem<N> left;
        f_combine<N>(*carry, tot[blk - 1], left);
        f_combine<N>(left, pre[c], o);
      } else {
        f_combine<N>(*carry, pre[c], o);
      }
#pragma unroll
      for (int k = 0; k < N; ++k) m[k] = o.b[k];
#pragma unroll
      for (int k = 0; k < N * N; ++k) C[k] = o.C[k];
    } else {
      fwd_start_state<N>(pre, c, tot, m, C);
    }
#pragma unroll
    for (int k = 0; k < N * N; ++k) W[k] = md.W[k];
    MvnPrepared<N> mvn;  // S = W * 1.0 at every step: factorised once per thread
    if (TR) {
      mvn.prepare(W);
      st |= mvn.st;
    }
    advance<N, true>(md.G, W, 1.0, m, C, an, Rn);
    SElem<N> sacc;  // unused (no smoother fold)
    bool shave = false;
    auto row = [&](int64_t r, double yv, const double *Ft) {
      FwdRow<N> o;
      const bool init = ki && r == 0;
      fwd_row<N, false>(md, Ft, W, init, yv, m, C, an, Rn, o, st, false, sacc, shave);
      if (init) return;
      if (TR) tr += mvn.eval(o.m, o.a);
      if (!isnan(yv)) {
        const double sd = sqrt(o.Q);
        const double dd = (yv - o.f) / sd;
        li += -dd * dd / 2.0 - log(sqrt(2.0 * 3.141592653589793) * sd);
      }
    };
    int64_t r = r0;
    if (VEC) {
      YGroup<true> yg;
      FGroup<N, true> fg;
      yg.start(y, r0, ki);
      if constexpr (FTV) fg.start(Fd, r0, ki);
      for (; r + kGrp <= r1; r += kGrp) {
        double yv[kGrp], fv[kGrp][N];
        yg.load(y, r, T, ki, yv);
        if constexpr (FTV) fg.load(Fd, r, T, ki, fv);
#pragma unroll
        for (int i = 0; i < kGrp; ++i) row(r + i, yv[i], FTV ? fv[i] : md.F);
      }
    }
    for (; r < r1; ++r) row(r, r >= ki ? y[r - ki] : 0.0, (FTV && r >= ki) ? Fd + (r - ki) * N : md.F);
    if (r1 == rows) {  // this thread owns row T: its state is the final filtered state
#pragma unroll
      for (int k = 0; k < N; ++k) last[k] = m[k];
#pragma unroll
      for (int k = 0; k < N * N; ++k) last[N + k] = C[k];
    }
  }
  s_tr[tid] = tr; s_in[tid] = li; s_st[tid] = st;
  __syncthreads();
#pragma unroll
  for (int off = kLlBlock / 2; off > 0; off >>= 1) {
    if (tid < off) {
      s_tr[tid] = s_tr[tid] + s_tr[tid + off];
      s_in[tid] = s_in[tid] + s_in[tid + off];
      s_st[tid] |= s_st[tid + off];
    }
    __syncthreads();
  }
  if (tid == 0) part[blockIdx.x] = LoglikPart{s_tr[0], s_in[0], s_st[0]};
}

// One block: thread i sums parts i, i + kLlFinish, ... in order, then the same fixed-order tree.
// Status as the sequential kernel: the bits the sweep raised, plus BDLM_ST_NONFINITE when the final
// filtered mean is not finite (C is not checked).  A chunk of a time-sharded series that does not
// hold row T passes last = nullptr; st_out receives the status as a double (the rank's partial vector).
__global__ void __launch_bounds__(kLlFinish)
loglik_finish_kernel(const LoglikPart *part, int64_t nparts, const double *last, int n, double *transition,
                     double *innovations, double *m_last, double *C_last, int32_t *status, double *st_out) {
  __shared__ double s_tr[kLlFinish], s_in[kLlFinish];
  __shared__ int s_st[kLlFinish];
  const int tid = threadIdx.x;
  double tr = 0.0, li = 0.0;
  int st = 0;
  for (int64_t i = tid; i < nparts; i += kLlFinish) {
    tr = tr + part[i].tr;
    li = li + part[i].in;
    st |= part[i].st;
  }
  s_tr[tid] = tr; s_in[tid] = li; s_st[tid] = st;
  __syncthreads();
#pragma unroll
  for (int off = kLlFinish / 2; off > 0; off >>= 1) {
    if (tid < off) {
      s_tr[tid] = s_tr[tid] + s_tr[tid + off];
      s_in[tid] = s_in[tid] + s_in[tid + off];
      s_st[tid] |= s_st[tid + off];
    }
    __syncthreads();
  }
  if (tid != 0) return;
  if (transition) *transition = s_tr[0];
  if (innovations) *innovations = s_in[0];
  bool finite = true;
  if (last) {
    for (int k = 0; k < n; ++k) {
      finite = finite && isfinite(last[k]);
      if (m_last) m_last[k] = last[k];
    }
    if (C_last)
      for (int k = 0; k < n * n; ++k) C_last[k] = last[n + k];
  }
  const int bits = s_st[0] | (finite ? 0 : BDLM_ST_NONFINITE);
  if (status) *status = bits;
  if (st_out) *st_out = (double)bits;
}

// bdlm_scan_dist_loglik_finish: every rank's [transition, innovations, status] partial vector, added
// in rank order by one thread, so every rank writes the same bits.
__global__ void dist_loglik_finish_kernel(const double *parts, int world, double *transition,
                                          double *innovations, int32_t *status) {
  double tr = 0.0, li = 0.0;
  int st = 0;
  for (int r = 0; r < world; ++r) {
    tr = tr + parts[3 * r];
    li = li + parts[3 * r + 1];
    st |= (int)parts[3 * r + 2];
  }
  if (transition) *transition = tr;
  if (innovations) *innovations = li;
  if (status) *status = st;
}

// ---- apply, backward: sequential (textbook) RTS recursion from the scanned successor state
template <int N>
__device__ __forceinline__ bool state_finite(const double *s, const double *S) {
  bool finite = true;
#pragma unroll
  for (int i = 0; i < N; ++i) finite = finite && isfinite(s[i]);
#pragma unroll
  for (int k = 0; k < N * N; ++k) finite = finite && isfinite(S[k]);
  return finite;
}

template <int N>
__device__ __forceinline__ void bwd_step(const ScanModel<N> &md, const double (&W)[N * N],
                                         const double (&m)[N], const double (&C)[N * N],
                                         double (&s)[N], double (&S)[N * N], int &st) {
  // textbook RTS step (small_steps.cuh rts_step) with the gain formed from one explicit inverse:
  //   B = C G^T R1^-1,  s = m + B (s - a1),  S = C - B (R1 - S) B^T
  double a1[N], R1[N * N], CGt[N * N], Rinv[N * N], Bg[N * N], d[N], t[N], Dm[N * N], t1[N * N], t2[N * N];
  advance<N, true>(md.G, W, 1.0, m, C, a1, R1);
  smm<N, N, N, false, true>(C, md.G, CGt);
  st |= small_inverse<N>(R1, Rinv);
  smm<N, N, N, false, false>(CGt, Rinv, Bg);
#pragma unroll
  for (int i = 0; i < N; ++i) d[i] = s[i] - a1[i];
  smm<N, N, 1, false, false>(Bg, d, t);
#pragma unroll
  for (int k = 0; k < N * N; ++k) Dm[k] = R1[k] - S[k];
  smm<N, N, N, false, false>(Bg, Dm, t1);
  smm<N, N, N, false, true>(t1, Bg, t2);
#pragma unroll
  for (int i = 0; i < N; ++i) s[i] = m[i] + t[i];
#pragma unroll
  for (int k = 0; k < N * N; ++k) S[k] = C[k] - t2[k];
}
template <int N, bool VEC>
__device__ __forceinline__ void bwd_row(const ScanModel<N> &md, const double (&W)[N * N], const View &fm,
                                        const View &fC, int64_t r, double (&s)[N], double (&S)[N * N],
                                        int &st) {
  double m[N], C[N * N];
  load_row<N, VEC>(fm, r, m);
  load_row<N * N, VEC>(fC, r, C);
  bwd_step<N>(md, W, m, C, s, S, st);
}

template <int N, bool VEC>
__global__ void __launch_bounds__(128, 1)
bwd_apply_kernel(const ScanModel<N> md, View fm, View fC, int64_t nrows, int64_t M,
                 const SElem<N> *suf /* [M+1] suffix-inclusive scan, slot M = terminal */,
                 View sv, View Sv, int32_t *status,
                 const SElem<N> *carry /* multi-GPU: everything after this chunk, or nullptr */,
                 const SElem<N> *tot /* scanned level-2 block totals (scan order) `suf` still lacks, or nullptr */,
                 int sub) {
  const int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (c >= M) return;
  const int64_t r0 = c * (int64_t)sub, r1 = (r0 + sub < nrows) ? r0 + sub : nrows;
  double W[N * N], s[N], S[N * N];
  int st = 0;
  const int64_t blk = (M - (c + 1)) / (kScanBlock * kPer);  // suffix scan: position = M - index
  const bool use_tot = tot && blk > 0;
  if (carry || use_tot) {
    SElem<N> o;
    if (carry && use_tot) {
      SElem<N> mid;
      s_combine<N>(suf[c + 1], tot[blk - 1], mid);  // later blocks of this chunk
      s_combine<N>(mid, *carry, o);                  // later chunks
    } else {
      s_combine<N>(suf[c + 1], carry ? *carry : tot[blk - 1], o);
    }
#pragma unroll
    for (int k = 0; k < N * N; ++k) S[k] = o.L[k];
#pragma unroll
    for (int k = 0; k < N; ++k) s[k] = o.g[k];
  } else {
#pragma unroll
    for (int k = 0; k < N * N; ++k) S[k] = suf[c + 1].L[k];
#pragma unroll
    for (int k = 0; k < N; ++k) s[k] = suf[c + 1].g[k];
  }
#pragma unroll
  for (int k = 0; k < N * N; ++k) W[k] = md.W[k];
  int64_t r = r1;  // one past the next row to produce
  // ragged head of the descending sweep (rows above the last whole group), scalar stores
  const int64_t aligned_top = VEC ? r0 + (r1 - r0) / kGrp * kGrp : r1;
  auto scalar_row = [&](int64_t row) {
    bwd_row<N, VEC>(md, W, fm, fC, row, s, S, st);
    store_row_scalar<N>(sv, row, s);
    store_row_scalar<N * N>(Sv, row, S);
  };
  if (VEC) {
    for (; r > aligned_top; --r) scalar_row(r - 1);
    for (; r - kGrp >= r0; r -= kGrp) {
      const int64_t g0 = r - kGrp;
      GroupBuf<N> gs;
      GroupBuf<N * N> gS;
      constexpr bool kGroupLoad = N <= 2;  // whole-line loads when the register budget allows
      double gm[kGrp * N], gC[kGrp * N * N];  // dead (eliminated) when !kGroupLoad
      if constexpr (kGroupLoad) {
        load_group<N>(fm, g0, gm);
        load_group<N * N>(fC, g0, gC);
      }
#define BDLM_BWD_ROW(I)                                                          \
  {                                                                              \
    if constexpr (kGroupLoad) {                                                  \
      double m_[N], C_[N * N];                                                   \
      for (int k = 0; k < N; ++k) m_[k] = gm[I * N + k];                         \
      for (int k = 0; k < N * N; ++k) C_[k] = gC[I * N * N + k];                 \
      bwd_step<N>(md, W, m_, C_, s, S, st);                                      \
    } else {                                                                     \
      bwd_row<N, VEC>(md, W, fm, fC, g0 + I, s, S, st);                          \
    }                                                                            \
    if (sv.ptr) gs.template put<I, false>(sv.ptr + g0 * N, s);                   \
    if (Sv.ptr) gS.template put<I, false>(Sv.ptr + g0 * (N * N), S);             \
  }
      BDLM_BWD_ROW(3) BDLM_BWD_ROW(2) BDLM_BWD_ROW(1) BDLM_BWD_ROW(0)
#undef BDLM_BWD_ROW
    }
  }
  for (; r > r0; --r) scalar_row(r - 1);
  // (s, S) now hold row 0 of the chunk.  For the whole series that is the smoothed initial state,
  // the final state of the sequential kernels, which flag it when it is not finite.
  if (c == 0 && !state_finite<N>(s, S)) st |= BDLM_ST_NONFINITE;
  if (status && st) atomicOr(status, st);
}

// ---- backward sampler + Gibbs statistics (bdlm_scan_ffbs) ------------------------------------
// On the regular grid Smoothing.step's draw (ffbs_small.cu) is affine in the successor draw:
//   theta_r = B_r theta_{r+1} + c_r,   c_r = m_r - B_r a_{r+1} + M_r z_r    (r < T)
//   theta_T = m_T + M_T z_T
// with B_r = C_r G^T R_{r+1}^-1 and M_r = V diag(sqrt(lam)) from jacobi_eigsym_small of the same
// symmetrised Joseph-form covariance H_r the sequential kernel forms.  The eigen basis is part of
// the contract: any other square root of H_r is an equally valid draw, but gives another path for
// the same z.  Elements (B_r, c_r) compose as the (E, g) part of SElem; a type of their own saves
// SElem's E L E^T (2 n^3 multiply-adds per combine) and a third of the level-2 shared memory.
template <int N>
struct BElem {
  double E[N * N], g[N];
};

// out = ei (x) ej, ei earlier:  E = E_i E_j ; g = E_i g_j + g_i
template <int N>
__host__ __device__ __forceinline__ void b_combine(const BElem<N> &ei, const BElem<N> &ej, BElem<N> &out) {
  double v[N];
  smm<N, N, N, false, false>(ei.E, ej.E, out.E);
  smm<N, N, 1, false, false>(ei.E, ej.g, v);
#pragma unroll
  for (int k = 0; k < N; ++k) out.g[k] = v[k] + ei.g[k];
}
template <int N>
__host__ __device__ __forceinline__ void b_identity(BElem<N> &e) {
#pragma unroll
  for (int k = 0; k < N * N; ++k) e.E[k] = (k % (N + 1) == 0) ? 1.0 : 0.0;
#pragma unroll
  for (int k = 0; k < N; ++k) e.g[k] = 0.0;
}
template <int N>
struct Op<BElem<N>> {
  __device__ static void apply(const BElem<N> &earlier, const BElem<N> &later, BElem<N> &o) {
    b_combine<N>(earlier, later, o);
  }
};

// Philox key of the on-device normals (z == NULL), as ffbs_small_kernel's.  The offset depends on the
// GLOBAL row and row count, so a chunk of a time-sharded series draws the normals the whole series
// would: local row r is global row first + r of rows.
struct FfbsRng {
  unsigned long long seed, sweep;
  long long base;         // subsequence of the series
  long long rows, first;  // global row count (T + 1) and global index of the chunk's row 0
};

// The n normals consumed for theta[row] (local row): injected, or Philox exactly as the sequential kernel
template <int N>
__device__ __forceinline__ void ffbs_normals(const CView &z, const FfbsRng &rng, int64_t row, double (&zr)[N]) {
  if (z.ptr) {
#pragma unroll
    for (int k = 0; k < N; ++k) zr[k] = ld_stream(z.ptr + row * z.sr + k * z.sk);
  } else {
    const RngKey key{rng.seed, rng.sweep};
#pragma unroll
    for (int k = 0; k < N; ++k) zr[k] = philox_normal(key, rng.base, (int)rng.rows, (int)(rng.first + row), N, k);
  }
}

// RTS gain of row r from its filtered (m, C): B = C G^T R1^-1 (one inverse, as bwd_step), and a1.
template <int N>
__device__ __forceinline__ void ffbs_gain(const ScanModel<N> &md, const double (&W)[N * N], const double (&m)[N],
                                          const double (&C)[N * N], double (&a1)[N], double (&Bg)[N * N],
                                          int &st) {
  double R1[N * N], CGt[N * N], Rinv[N * N];
  advance<N, true>(md.G, W, 1.0, m, C, a1, R1);
  smm<N, N, N, false, true>(C, md.G, CGt);
  st |= small_inverse<N>(R1, Rinv);
  smm<N, N, N, false, false>(CGt, Rinv, Bg);
}

// Element (B_r, c_r) of a row with a successor.  H_r = (I - B G) C (I - B G)^T + B W B^T,
// symmetrised, as Smoothing.step (:93-95) and ffbs_small_kernel form it.
template <int N>
__device__ __forceinline__ void ffbs_element(const ScanModel<N> &md, const double (&W)[N * N], const double (&m)[N],
                                             const double (&C)[N * N], const double (&z)[N], double (&Bg)[N * N],
                                             double (&cr)[N], int &st) {
  double a1[N], v[N], g[N], D[N * N], t1[N * N], t2[N * N], Hm[N * N], Hs[N * N];
  ffbs_gain<N>(md, W, m, C, a1, Bg, st);
  smm<N, N, 1, false, false>(Bg, a1, v);
#pragma unroll
  for (int i = 0; i < N; ++i) g[i] = m[i] - v[i];
  smm<N, N, N, false, false>(Bg, md.G, D);
#pragma unroll
  for (int j = 0; j < N; ++j)
#pragma unroll
    for (int i = 0; i < N; ++i) D[i + j * N] = ((i == j) ? 1.0 : 0.0) - D[i + j * N];
  smm<N, N, N, false, false>(D, C, t1);
  smm<N, N, N, false, true>(t1, D, Hm);
  smm<N, N, N, false, false>(Bg, W, t1);
  smm<N, N, N, false, true>(t1, Bg, t2);
#pragma unroll
  for (int k = 0; k < N * N; ++k) Hm[k] = Hm[k] + t2[k];
#pragma unroll
  for (int j = 0; j < N; ++j)
#pragma unroll
    for (int i = 0; i < N; ++i) Hs[i + j * N] = (Hm[i + j * N] + Hm[j + i * N]) / 2.0;
  st |= eig_draw_small<N>(g, Hs, z, cr);
}

// Level 1 of the sampler: thread c owns rows [c*sub, min((c+1)*sub, T)) -- the smoother's row
// ownership -- and folds their elements in descending order.  c_r goes to theta's own row r as
// scratch, so the apply sweep reads it back instead of repeating the eigen-decomposition.  The
// thread that owns row T - 1 also draws theta_T and writes the terminal element (0, theta_T) when
// row T is the series' last (term = T; a chunk of a time-sharded series that others follow passes
// term = -1 and its caller sets the terminal slot to the identity).
template <int N, bool VEC>
__global__ void __launch_bounds__(128)
ffbs_reduce_kernel(const ScanModel<N> md, View fm, View fC, int64_t T, int64_t M, CView z, FfbsRng rng,
                   View th, BElem<N> *agg /* [M + 1], slot M = terminal */, int32_t *status, int sub,
                   int64_t term) {
  const int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (c >= M) return;
  const int64_t r0 = c * (int64_t)sub, r1 = (r0 + sub < T) ? r0 + sub : T;
  double W[N * N];
#pragma unroll
  for (int k = 0; k < N * N; ++k) W[k] = md.W[k];
  int st = 0;
  if (r1 == term) {  // Smoothing.initialise: theta_T ~ N(m_T, C_T)
    double m[N], C[N * N], zr[N], tT[N];
    load_row<N, false>(fm, T, m);
    load_row<N * N, false>(fC, T, C);
    ffbs_normals<N>(z, rng, T, zr);
    st |= eig_draw_small<N>(m, C, zr, tT);
    store_row_scalar<N>(th, T, tT);
    BElem<N> e;
#pragma unroll
    for (int k = 0; k < N * N; ++k) e.E[k] = 0.0;
#pragma unroll
    for (int k = 0; k < N; ++k) e.g[k] = tT[k];
    agg[M] = e;
  }
  BElem<N> acc;
  bool have = false;
  auto fold = [&](int64_t r, double (&cr)[N]) {
    double m[N], C[N * N], zr[N];
    BElem<N> e, o;
    load_row<N, VEC>(fm, r, m);
    load_row<N * N, VEC>(fC, r, C);
    ffbs_normals<N>(z, rng, r, zr);
    ffbs_element<N>(md, W, m, C, zr, e.E, e.g, st);
#pragma unroll
    for (int k = 0; k < N; ++k) cr[k] = e.g[k];
    if (have) { b_combine<N>(e, acc, o); acc = o; }
    else { acc = e; have = true; }
  };
  // Whole-sector group stores for n <= 3 (a row of n = 4 is one sector already): four inlined
  // eigen-decompositions of n = 4 would spill.
  constexpr bool kGroupStore = VEC && N <= 3;
  int64_t r = r1;
  const int64_t aligned_top = kGroupStore ? r0 + (r1 - r0) / kGrp * kGrp : r1;
  auto scalar_row = [&](int64_t row) {
    double cr[N];
    fold(row, cr);
    store_row_scalar<N>(th, row, cr);
  };
  if constexpr (kGroupStore) {
    for (; r > aligned_top; --r) scalar_row(r - 1);
    for (; r - kGrp >= r0; r -= kGrp) {
      const int64_t g0 = r - kGrp;
      GroupBuf<N> gc;
#define BDLM_FFBS_FOLD(I)                               \
  {                                                     \
    double cr[N];                                       \
    fold(g0 + I, cr);                                   \
    gc.template put<I, false>(th.ptr + g0 * N, cr);     \
  }
      BDLM_FFBS_FOLD(3) BDLM_FFBS_FOLD(2) BDLM_FFBS_FOLD(1) BDLM_FFBS_FOLD(0)
#undef BDLM_FFBS_FOLD
    }
  }
  for (; r > r0; --r) scalar_row(r - 1);
  agg[c] = acc;
  if (status && st) atomicOr(status, st);
}

// Gibbs statistics of one path (ffbs_small_kernel / oracle_gibbs_stats), dt = 1:
// [ssy, ny, ssw[N], scatter[N*N]]
template <int N>
struct FfbsStats {
  static constexpr int kD = 2 + N + N * N;
  double v[kD];
  __device__ __forceinline__ void zero() {
#pragma unroll
    for (int k = 0; k < kD; ++k) v[k] = 0.0;
  }
  // step t: theta_{t+1} = cur, theta_t = prev, observation y_t with F = F_t.  The observation term needs
  // theta_{t+1} alone, the transition term both: a time-sharded chunk counts them on different rows.
  __device__ __forceinline__ void add_obs(const double *F, const double (&cur)[N], double yt) {
    double ft;
    smm<1, N, 1, true, false>(F, cur, &ft);
    if (!isnan(yt)) {
      v[0] = v[0] + (yt - ft) * (yt - ft);
      v[1] = v[1] + 1.0;
    }
  }
  __device__ __forceinline__ void add_trans(const ScanModel<N> &md, const double (&cur)[N], const double (&prev)[N]) {
    double gx[N], diff[N];
    smm<N, N, 1, false, false>(md.G, prev, gx);
#pragma unroll
    for (int i = 0; i < N; ++i) diff[i] = cur[i] - gx[i];
#pragma unroll
    for (int i = 0; i < N; ++i) v[2 + i] = v[2 + i] + diff[i] * diff[i];
#pragma unroll
    for (int j = 0; j < N; ++j)
#pragma unroll
      for (int i = 0; i < N; ++i) v[2 + N + i + j * N] = v[2 + N + i + j * N] + diff[i] * diff[j];
  }
};
constexpr int kFbBlock = 128, kFbFinish = 256;

// Apply: thread c takes its successor theta_{r1} (the scanned suffix composed with the deferred
// top-level block total and, on a chunk of a time-sharded series that others follow, the carry of
// the later chunks, as bwd_apply_kernel) and walks theta_r = B_r theta_{r+1} + c_r down its rows,
// c_r read back from theta's row r.  STATS: every row r it produces adds the transition term of the
// step theta_r -> theta_{r+1} (the last row of a chunk pairs with the carry's theta) and one
// observation term: with keep_init (the whole series, or rank 0) that of row r + 1, y[r], which
// belongs to the next chunk when r is the chunk's last row (y[r] does not exist: skipped); without
// it (ranks > 0) that of row r itself, y[r], plus that of the terminal row on the last chunk.  So
// every step and every observation is counted once across threads and ranks.  The block's sums go
// through a fixed-order shared-memory tree to one partial per block.  FTV: the observation term of
// y[r] uses F[r] = Fd + r*N (F is indexed like y).
template <int N, bool VEC, bool STATS, bool FTV = false>
__global__ void __launch_bounds__(kFbBlock, 1)
ffbs_apply_kernel(const ScanModel<N> md, View fm, View fC, const double *__restrict__ y, int64_t T, int64_t M,
                  const BElem<N> *suf /* [M+1] suffix-inclusive scan, slot M = terminal */,
                  const BElem<N> *tot /* scanned level-2 block totals (scan order) `suf` still lacks, or nullptr */,
                  View th, int32_t *status, int sub, double *part /* [kD][gridDim.x] */,
                  const BElem<N> *carry /* multi-GPU: everything after this chunk, or nullptr */,
                  int keep_init, int64_t ny /* observations in y */, bool terminal,
                  const double *__restrict__ Fd /* FTV: [ny][N] */) {
  constexpr int kD = FfbsStats<N>::kD;
  __shared__ double s_part[STATS ? kD * kFbBlock : 1];
  const int tid = threadIdx.x;
  const int64_t c = blockIdx.x * (int64_t)blockDim.x + tid;
  FfbsStats<N> acc;
  acc.zero();
  if (c < M) {
    const int64_t r0 = c * (int64_t)sub, r1 = (r0 + sub < T) ? r0 + sub : T;
    double W[N * N], t[N];
    int st = 0;
    const int64_t blk = (M - (c + 1)) / (kScanBlock * kPer);  // suffix scan: position = M - index
    const bool use_tot = tot && blk > 0;
    if (carry || use_tot) {
      BElem<N> o;
      if (carry && use_tot) {
        BElem<N> mid;
        b_combine<N>(suf[c + 1], tot[blk - 1], mid);  // later blocks of this chunk
        b_combine<N>(mid, *carry, o);                  // later chunks
      } else {
        b_combine<N>(suf[c + 1], carry ? *carry : tot[blk - 1], o);
      }
#pragma unroll
      for (int k = 0; k < N; ++k) t[k] = o.g[k];
    } else {
#pragma unroll
      for (int k = 0; k < N; ++k) t[k] = suf[c + 1].g[k];
    }
#pragma unroll
    for (int k = 0; k < N * N; ++k) W[k] = md.W[k];
    if (STATS && !keep_init && terminal && r1 == T)  // t = theta of the terminal row
      acc.add_obs(FTV ? Fd + T * N : md.F, t, y[T]);
    // theta_r from theta_{r+1} = t and c_r; t becomes theta_r
    auto step = [&](int64_t r, const double (&cr)[N], double yr, const double *Fr) {
      double m[N], C[N * N], a1[N], Bg[N * N], v[N], nt[N];
      load_row<N, VEC>(fm, r, m);
      load_row<N * N, VEC>(fC, r, C);
      ffbs_gain<N>(md, W, m, C, a1, Bg, st);
      smm<N, N, 1, false, false>(Bg, t, v);
#pragma unroll
      for (int k = 0; k < N; ++k) nt[k] = v[k] + cr[k];
      if (STATS) {
        if (keep_init) acc.add_obs(Fr, t, yr);
        else acc.add_obs(Fr, nt, yr);
        acc.add_trans(md, t, nt);
      }
#pragma unroll
      for (int k = 0; k < N; ++k) t[k] = nt[k];
    };
    int64_t r = r1;
    // group loads of y need y[g0 .. g0 + kGrp) to exist: rows at or above ny go the scalar way
    const int64_t vtop = (STATS && r1 > ny) ? ny : r1;
    const int64_t aligned_top = VEC ? r0 + (vtop - r0) / kGrp * kGrp : r1;
    auto scalar_row = [&](int64_t row) {
      double cr[N];
      load_row<N, false>(th, row, cr);
      step(row, cr, STATS ? (row < ny ? y[row] : __longlong_as_double(0x7ff8000000000000LL)) : 0.0,
           (FTV && row < ny) ? Fd + row * N : md.F);
      store_row_scalar<N>(th, row, t);
    };
    if (VEC) {
      for (; r > aligned_top; --r) scalar_row(r - 1);
      for (; r - kGrp >= r0; r -= kGrp) {
        const int64_t g0 = r - kGrp;
        double cg[kGrp * N], yg[kGrp], fg[kGrp * N];
        load_group<N>(th, g0, cg);  // every c of the group before the first store into it
        if (STATS) ld_v4(y + g0, yg);
        if constexpr (STATS && FTV) {
#pragma unroll
          for (int k = 0; k < kGrp * N; k += 4) ld_v4(Fd + g0 * N + k, fg + k);
        }
        GroupBuf<N> gt;
#define BDLM_FFBS_APPLY(I)                                 \
  {                                                        \
    double cr[N];                                          \
    for (int k = 0; k < N; ++k) cr[k] = cg[I * N + k];     \
    step(g0 + I, cr, STATS ? yg[I] : 0.0, FTV ? fg + I * N : md.F); \
    gt.template put<I, false>(th.ptr + g0 * N, t);         \
  }
        BDLM_FFBS_APPLY(3) BDLM_FFBS_APPLY(2) BDLM_FFBS_APPLY(1) BDLM_FFBS_APPLY(0)
#undef BDLM_FFBS_APPLY
      }
    }
    for (; r > r0; --r) scalar_row(r - 1);
    // t is theta_{r0}; for thread 0 of the series' first chunk the final state of the sequential
    // sampler, flagged likewise
    if (c == 0 && keep_init) {
      bool finite = true;
#pragma unroll
      for (int k = 0; k < N; ++k) finite = finite && isfinite(t[k]);
      if (!finite) st |= BDLM_ST_NONFINITE;
    }
    if (status && st) atomicOr(status, st);
  }
  if constexpr (STATS) {
#pragma unroll
    for (int k = 0; k < kD; ++k) s_part[k * kFbBlock + tid] = acc.v[k];
    __syncthreads();
#pragma unroll
    for (int off = kFbBlock / 2; off > 0; off >>= 1) {
      if (tid < off) {
#pragma unroll
        for (int k = 0; k < kD; ++k)
          s_part[k * kFbBlock + tid] = s_part[k * kFbBlock + tid] + s_part[k * kFbBlock + tid + off];
      }
      __syncthreads();
    }
    if (tid < kD) part[(int64_t)tid * gridDim.x + blockIdx.x] = s_part[tid * kFbBlock];
  }
}

// One block: thread i sums partials i, i + kFbFinish, ... of each statistic in order, then the
// same fixed-order tree; no atomics, so a call gives the same bits on any stream or context.
// vec (a chunk of a time-sharded series): the sums and then the chunk's status bits go to the rank's
// partial vector [kD + 1] instead of sv.
template <int N>
__global__ void __launch_bounds__(kFbFinish)
ffbs_stats_finish_kernel(const double *part, int64_t nparts, StatViews sv, double *vec, const int32_t *status) {
  constexpr int kD = FfbsStats<N>::kD;
  __shared__ double s[kFbFinish];
  const int tid = threadIdx.x;
  for (int k = 0; k < kD; ++k) {
    double x = 0.0;
    for (int64_t i = tid; i < nparts; i += kFbFinish) x = x + part[(int64_t)k * nparts + i];
    s[tid] = x;
    __syncthreads();
    for (int off = kFbFinish / 2; off > 0; off >>= 1) {
      if (tid < off) s[tid] = s[tid] + s[tid + off];
      __syncthreads();
    }
    if (tid == 0) {
      const double v = s[0];
      if (vec) vec[k] = v;
      else if (k == 0) { if (sv.ssy.ptr) sv.ssy.ptr[0] = v; }
      else if (k == 1) { if (sv.ny.ptr) sv.ny.ptr[0] = v; }
      else if (k < 2 + N) { if (sv.ssw.ptr) sv.ssw.ptr[(k - 2) * sv.ssw.sk] = v; }
      else if (sv.scatter.ptr) sv.scatter.ptr[(k - 2 - N) * sv.scatter.sk] = v;
    }
    __syncthreads();
  }
  if (vec && tid == 0) vec[kD] = status ? (double)*status : 0.0;
}

// bdlm_scan_dist_ffbs_stats_finish: every rank's partial vector [ssy, ny, ssw, scatter, status],
// added in rank order by one thread, so every rank writes the same bits.
template <int N>
__global__ void dist_ffbs_stats_finish_kernel(const double *parts, int world, StatViews sv, int32_t *status) {
  constexpr int kD = FfbsStats<N>::kD;
  int st = 0;
  for (int r = 0; r < world; ++r) st |= (int)parts[r * (kD + 1) + kD];
  for (int k = 0; k < kD; ++k) {
    double v = 0.0;
    for (int r = 0; r < world; ++r) v = v + parts[r * (kD + 1) + k];
    if (k == 0) { if (sv.ssy.ptr) sv.ssy.ptr[0] = v; }
    else if (k == 1) { if (sv.ny.ptr) sv.ny.ptr[0] = v; }
    else if (k < 2 + N) { if (sv.ssw.ptr) sv.ssw.ptr[(k - 2) * sv.ssw.sk] = v; }
    else if (sv.scatter.ptr) sv.scatter.ptr[(k - 2 - N) * sv.scatter.sk] = v;
  }
  if (status) *status = st;
}

// terminal slot of a chunk that others follow: the identity, so that the chunk's aggregate leaves
// them out (the finish phase brings them in through the carry)
template <int N>
__global__ void set_s_identity(SElem<N> *slot) {
  SElem<N> e;
  s_identity<N>(e);
  *slot = e;
}
template <int N>
__global__ void set_b_identity(BElem<N> *slot) {
  BElem<N> e;
  b_identity<N>(e);
  *slot = e;
}
// last chunk: s_T = m_T, S_T = C_T go to the outputs and become the terminal element of the scan.
// status: the row is also row 0 (a single row, no backward sweep follows): flag it as that sweep would.
template <int N>
__global__ void terminal_from_last_row(View fm, View fC, int64_t row, View sv, View Sv, SElem<N> *slot,
                                       int32_t *status) {
  double sS[N + N * N];
  for (int k = 0; k < N; ++k) {
    const double v = fm.ptr[row * fm.sr + k * fm.sk];
    if (sv.ptr) sv.ptr[row * sv.sr + k * sv.sk] = v;
    sS[k] = v;
  }
  for (int k = 0; k < N * N; ++k) {
    const double v = fC.ptr[row * fC.sr + k * fC.sk];
    if (Sv.ptr) Sv.ptr[row * Sv.sr + k * Sv.sk] = v;
    sS[N + k] = v;
  }
  if (status && !state_finite<N>(sS, sS + N)) atomicOr(status, BDLM_ST_NONFINITE);
  SElem<N> e;
  s_state<N>(e, sS, sS + N);
  *slot = e;
}

// ---- peer-mailbox exchange of the chunk aggregates (single-process communicators, comm.cu) ----
// Publish: block d stores this rank's aggregate into slot [rank] of rank d's box with plain 8-byte
// stores over NVLink (or locally for d == rank), fences at system scope, then one thread releases
// flag[d][rank] = epoch.  One launch replaces the device-to-device copy + the NCCL all-gather.
template <class E>
__global__ void __launch_bounds__(64)
publish_kernel(const E *src, const ScanPeers peers, int rank, const unsigned long long *epoch_dev) {
  constexpr int kD = (int)(sizeof(E) / sizeof(double));
  const int d = blockIdx.x;
  const double *s = reinterpret_cast<const double *>(src);
  double *dst = peers.box[d] + (size_t)rank * kD;
  for (int k = threadIdx.x; k < kD; k += blockDim.x) dst[k] = s[k];
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    volatile unsigned long long *f = peers.flag[d] + rank;
    *f = *epoch_dev;  // this device's call counter (bumped by epoch_bump_kernel at the start of a call)
  }
}

// Acquire side: spin (bounded -- a peer that died must not hang this GPU) until the slot of
// `src_rank` in MY box carries this call's epoch, then read it with volatile loads.
constexpr int kPeerSpinMax = 1 << 24;
template <class E>
__device__ bool peer_wait_read(const ScanPeers &peers, int my_rank, int src_rank,
                               const unsigned long long *epoch_dev, E &out) {
  const unsigned long long epoch = *epoch_dev;
  constexpr int kD = (int)(sizeof(E) / sizeof(double));
  volatile unsigned long long *f = peers.flag[my_rank] + src_rank;
  int spins = 0;
  while (*f < epoch) {
    if (++spins > kPeerSpinMax) return false;
    __nanosleep(64);
  }
  __threadfence_system();
  const volatile double *s = peers.box[my_rank] + (size_t)src_rank * kD;
  double *o = reinterpret_cast<double *>(&out);
  for (int k = 0; k < kD; ++k) o[k] = s[k];
  return true;
}

// Carry folding on the device (multi-GPU): one thread, at most world - 1 combines.  The aggregates
// come from `aggs` (NCCL all-gather already done on this stream) or, with peers.world > 0, from
// this rank's mailbox as the peers publish them.
template <int N>
__global__ void fold_forward_kernel(const FElem<N> *aggs, int rank, const StateArg<N> prior,
                                    FElem<N> *carry, const ScanPeers peers,
                                    const unsigned long long *epoch, int32_t *status) {
  FElem<N> e, t, in;
  f_state<N>(e, prior.v, prior.v + N);  // the state before the first observation of rank 0
  for (int r = 0; r < rank; ++r) {
    if (peers.world > 0) {
      if (!peer_wait_read(peers, rank, r, epoch, in)) { if (status) atomicOr(status, BDLM_ST_TIMEOUT); break; }
    } else {
      in = aggs[r];
    }
    f_combine<N>(e, in, t); e = t;
  }
  *carry = e;
}
// carry of rank r = agg_{r+1} (x) ... (x) agg_{world-1}; the last rank's aggregate already ends in
// its terminal state s_T = m_T, S_T = C_T.
template <int N>
__global__ void fold_backward_kernel(const SElem<N> *aggs, int rank, int world, SElem<N> *carry,
                                     const ScanPeers peers, const unsigned long long *epoch,
                                     int32_t *status) {
  SElem<N> e, t, in;
  bool ok = true;
  if (peers.world > 0) ok = peer_wait_read(peers, rank, world - 1, epoch, e);
  else e = aggs[world - 1];
  for (int r = world - 2; r > rank && ok; --r) {
    if (peers.world > 0) ok = peer_wait_read(peers, rank, r, epoch, in);
    else in = aggs[r];
    if (ok) { s_combine<N>(in, e, t); e = t; }
  }
  if (!ok && status) atomicOr(status, BDLM_ST_TIMEOUT);
  *carry = e;
}

// carry of rank r for the sampler: agg_{r+1} (x) ... (x) agg_{world-1} (rank < world - 1).  The last
// rank's aggregate ends in its terminal element (0, theta_T), so E = 0 and g is theta at the first row
// of chunk r + 1.
template <int N>
__global__ void fold_sampler_kernel(const BElem<N> *aggs, int rank, int world, BElem<N> *carry) {
  BElem<N> e = aggs[world - 1], t;
  for (int r = world - 2; r > rank; --r) { b_combine<N>(aggs[r], e, t); e = t; }
  *carry = e;
}

// ---- rows per thread (level-1 granularity), chosen per call ------------------------------------
// The two apply sweeps are register-heavy (3 resident blocks of 128 threads per SM for n = 2), so
// their time goes in WAVES of `slots` blocks, each as long as one thread's `sub` rows; the level-2
// scan costs per element, i.e. per T / sub.  A fixed 64 rows per thread left 2^22 rows with 512
// blocks for 444 slots (a second, almost empty wave) and 2^21 rows with every thread serially
// walking 64 rows on a 58 % occupied GPU.  Cost model fitted on B200 (profiles/r2_tuning.txt).
template <int N>
int apply_slots() {
  static const int slots = [] {  // devices of one process are alike
    int dev = 0, sms = 0, bf = 0, bb = 0;
    if (cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bf, fwd_apply_kernel<N, true, true>, 128, 0) != cudaSuccess ||
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bb, bwd_apply_kernel<N, true>, 128, 0) != cudaSuccess) {
      cudaGetLastError();
      return 148 * 2;
    }
    const int b = bf < bb ? bf : bb;
    return sms * (b < 1 ? 1 : b);
  }();
  return slots;
}

// f(std::integral_constant<int, N>{}) for the scan's state dimension n = N (1..4), else `none`.
template <class R, class F>
R with_n(int n, R none, F &&f) {
  switch (n) {
    case 1: return f(std::integral_constant<int, 1>{});
    case 2: return f(std::integral_constant<int, 2>{});
    case 3: return f(std::integral_constant<int, 3>{});
    case 4: return f(std::integral_constant<int, 4>{});
    default: return none;
  }
}

// f(std::bool_constant<b>...) for the run-time flags b...: one kernel instance per combination.
template <class F>
void with_flags(F &&f) { f(); }
template <class F, class... Bs>
void with_flags(F &&f, bool b, Bs... bs) {
  if (b) with_flags([&](auto... x) { f(std::true_type{}, x...); }, bs...);
  else with_flags([&](auto... x) { f(std::false_type{}, x...); }, bs...);
}

int scan_rows_per_thread(int n, int64_t T) {
  const int slots = with_n(n, 444, [](auto N) { return apply_slots<N>(); });
  const double rows = (double)(T + 1);
  int best = kSub;
  double best_cost = 1e300;
  // multiples of 16 rows only: a thread's run of every output field then starts on a 128-byte line
  // even for n = 1 (8 bytes per row); 60 rows per thread cost n = 1 13 % (lines shared by two threads)
  for (int sub = 16; sub <= kSub; sub += 16) {
    const double blocks = std::ceil(rows / (sub * 128.0));
    const double waves = blocks / slots;
    // a partly filled last wave is cheaper than a full one where the sweep is throughput-bound,
    // as long where it is latency-bound: take the middle
    const double sweep = 3.1 * sub * 0.5 * (std::ceil(waves) + waves);  // us
    const double level2 = 0.00057 * rows / sub;                         // us
    const double cost = sweep + level2;
    if (cost < best_cost) { best_cost = cost; best = sub; }
  }
  return best;
}

// ---- geometry and workspace layout of one pass over a chunk ------------------------------------
enum ScanPass { kPassForward, kPassLoglik, kPassBackward, kPassSampler };

// `sub` rows per thread over the `rows` the sweep walks, M level-1 threads (their elements X[0, M),
// then the slot X[M]), the apply grid for the pass's block size and the level-2 blocks over
// X[0, M].  A finish phase finds its local phase's prefixes where this puts them because both
// derive the geometry here from the same chunk.
struct ScanGeom {
  int sub;
  int64_t rows, M, nb;
  unsigned blocks;
};
ScanGeom scan_geom(int n, int64_t T, int keep_init, bool has_successor, ScanPass pass) {
  ScanGeom g;
  g.sub = scan_rows_per_thread(n, T);
  // the forward passes walk every row, the backward ones the rows with a successor in the chunk
  const bool forward = pass == kPassForward || pass == kPassLoglik;
  g.rows = T + keep_init - (forward || has_successor ? 0 : 1);
  g.M = (g.rows + g.sub - 1) / g.sub;
  if (pass == kPassSampler && g.M < 1) g.M = 1;  // the last chunk may hold a single row
  const int block = pass == kPassLoglik ? kLlBlock : pass == kPassSampler ? kFbBlock : 128;
  g.blocks = (unsigned)((g.M + block - 1) / block);
  g.nb = (g.M + 1 + kScanBlock * kPer - 1) / (kScanBlock * kPer);
  return g;
}
ScanGeom scan_geom(const ScanArgs &a, ScanPass pass) {
  return scan_geom(a.n, a.T, a.keep_init, a.has_successor != 0, pass);
}

// Block totals device_scan leaves after the `count` elements it scans, over all its levels.
int64_t level2_elems(int64_t count) {
  constexpr int64_t per_block = kScanBlock * kPer;
  int64_t s = 0;
  for (int64_t nb = (count + per_block - 1) / per_block; nb > 1; nb = (nb + per_block - 1) / per_block) s += nb;
  return s;
}

// Workspace of one pass: X [M + 1], the level-2 block totals, and the carry of the other chunks.
template <class E>
struct ScanLayout {
  E *X, *scratch, *carry;
  ScanLayout(const ScanGeom &g, void *base)
      : X(reinterpret_cast<E *>(base)), scratch(X + (g.M + 1)), carry(scratch + level2_elems(g.M + 1)) {}
  static size_t bytes(const ScanGeom &g) { return sizeof(E) * (size_t)(g.M + 2 + level2_elems(g.M + 1)); }
};

template <int N>
ScanModel<N> make_model(const ScanArgs &a) {
  ScanModel<N> md;
  for (int k = 0; k < N * N; ++k) { md.G[k] = a.G[k]; md.W[k] = a.W[k]; }
  for (int k = 0; k < N; ++k) md.F[k] = a.F ? a.F[k] : 0.0;  // f_tv: the kernels read a.Fd
  md.V = a.V;
  return md;
}

#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return e_; } while (0)

// 256-bit path: dense rows (sk = 1, sr = K) on a 32-byte aligned base.
static bool dense_aligned(const View &v, int64_t K) {
  return !v.ptr || (v.sk == 1 && v.sr == K && (reinterpret_cast<uintptr_t>(v.ptr) & 31) == 0);
}

// 256-bit loads of the streamed inputs: y and, with f_tv, F on 32-byte aligned bases.
static bool inputs_aligned(const ScanArgs &a) {
  return ((reinterpret_cast<uintptr_t>(a.y) | reinterpret_cast<uintptr_t>(a.Fd)) & 31) == 0;
}

// The model's level-1 table, rebuilt on the host and uploaded when the model changed since the
// context last built it.
template <int N>
cudaError_t fwd_table_upload(const ScanArgs &a, const ScanModel<N> &md, cudaStream_t stream) {
  if (!a.table_upload) return cudaSuccess;
  static_assert(sizeof(FwdTable<N>) <= kScanTableBytes, "table buffer too small");
  FwdTable<N> host;
  build_fwd_table<N>(md, host);
  // pageable source: staged by the driver before the call returns
  return cudaMemcpyAsync(a.table, &host, sizeof(host), cudaMemcpyHostToDevice, stream);
}

// Level 1 + level 2 of the forward pass: X[0, M] = inclusive prefixes of (slot 0, aggregates) with
// the top level's block prefixes left in scratch (defer_top).  identity: slot 0 is the identity
// (chunk aggregate only), else the state st0 before the first observation.
template <int N>
cudaError_t fwd_prefixes(const ScanArgs &a, const ScanModel<N> &md, const ScanGeom &g, const ScanLayout<FElem<N>> &w,
                         const StateArg<N> &st0, bool identity, cudaStream_t stream, int64_t *launches) {
  const FwdTable<N> *tb = reinterpret_cast<const FwdTable<N> *>(a.table);
  const unsigned blocks = (unsigned)((g.M + 127) / 128);
  with_flags([&](auto VEC_, auto FTV_) {
    fwd_reduce_kernel<N, VEC_, FTV_><<<blocks, 128, 0, stream>>>(md, tb, a.y, a.T, g.M, a.keep_init, w.X, st0,
                                                                 identity, g.sub, a.Fd);
  }, inputs_aligned(a), a.Fd != nullptr);
  ++*launches;
  CK(cudaGetLastError());
  return device_scan<FElem<N>, false, false>(w.X, g.M + 1, w.scratch, stream, launches, /*defer_top=*/true);
}

template <int N>
cudaError_t scan_forward(const ScanArgs &a, cudaStream_t stream, int64_t *launches) {
  const ScanModel<N> md = make_model<N>(a);
  const ScanGeom g = scan_geom(a, kPassForward);
  const ScanLayout<FElem<N>> w(g, a.workspace);
  CK(fwd_table_upload<N>(a, md, stream));
  const bool local = a.phase == kScanDistLocal, finish = a.phase == kScanDistFinish;
  if (!finish) {
    // dist local: chunk aggregate only (identity start); apply: prefix of
    // (start (x) aggregates), a.start = host (m, C) of the state before t = 0
    const StateArg<N> st0 = state_arg<N>(local ? nullptr : a.start);
    CK(fwd_prefixes<N>(a, md, g, w, st0, local, stream, launches));
    // the whole chunk: last element of a one-block scan, else the last scanned block total
    const FElem<N> *whole = g.nb > 1 ? w.scratch + (g.nb - 1) : w.X + g.M;
    if (local) {
      if (a.peers.world > 0) {  // straight into every peer's mailbox over NVLink
        publish_kernel<FElem<N>><<<a.peers.world, 64, 0, stream>>>(whole, a.peers, a.rank, a.epoch_dev);
        ++*launches;
        return cudaGetLastError();
      }
      // stays on the device: the caller all-gathers it (NCCL) on the same stream
      return cudaMemcpyAsync(a.agg_dev, whole, sizeof(FElem<N>), cudaMemcpyDeviceToDevice, stream);
    }
  } else {
    // X still holds this rank's scanned prefixes from the local phase
    fold_forward_kernel<N><<<1, 1, 0, stream>>>(reinterpret_cast<const FElem<N> *>(a.aggs_dev),
                                                a.rank, state_arg<N>(a.start), w.carry, a.peers,
                                                a.epoch_dev, a.status);
    ++*launches;
  }
  const bool vec = dense_aligned(a.kf.m, N) && dense_aligned(a.kf.C, N * N) &&
                   dense_aligned(a.kf.a, N) && dense_aligned(a.kf.R, N * N) &&
                   dense_aligned(a.kf.f, 1) && dense_aligned(a.kf.Q, 1) && inputs_aligned(a);
  // a.fuse_sagg: the caller runs the smoother next on the same rows: fold the smoothing
  // elements here so the backward pass starts from ready level-1 aggregates.
  SElem<N> *sagg = reinterpret_cast<SElem<N> *>(a.fuse_sagg);
  const int64_t nrows = scan_geom(a, kPassBackward).rows;  // the smoother's rows
  const FElem<N> *cr = finish ? w.carry : nullptr;
  const FElem<N> *tot = g.nb > 1 ? w.scratch : nullptr;  // top-level block prefixes, composed by the sweep
  with_flags([&](auto VEC_, auto FUSE_, auto FTV_) {
    fwd_apply_kernel<N, VEC_, FUSE_, FTV_><<<g.blocks, 128, 0, stream>>>(md, a.y, a.T, g.M, w.X, a.keep_init, a.kf,
                                                                        a.status, sagg, nrows, cr, tot, g.sub, a.Fd);
  }, vec, sagg != nullptr, a.Fd != nullptr);
  ++*launches;
  return cudaGetLastError();
}

// Log-likelihoods + last filtered state of the whole series (keep_init = 1): reduce, level-2 scan,
// the store-free sweep and the fixed-order sum of its block partials.
template <int N>
cudaError_t scan_loglik(const ScanArgs &a, const ScanLoglikOut &o, cudaStream_t stream, int64_t *launches) {
  if (a.keep_init != 1 || a.phase != kScanApply) return cudaErrorInvalidValue;
  const ScanModel<N> md = make_model<N>(a);
  const ScanGeom g = scan_geom(a, kPassLoglik);
  const ScanLayout<FElem<N>> w(g, a.workspace);
  LoglikPart *part = reinterpret_cast<LoglikPart *>(o.parts);
  double *last = reinterpret_cast<double *>(part + g.blocks);
  CK(fwd_table_upload<N>(a, md, stream));
  CK(fwd_prefixes<N>(a, md, g, w, state_arg<N>(a.start), false, stream, launches));
  const FElem<N> *tot = g.nb > 1 ? w.scratch : nullptr;
  with_flags([&](auto VEC_, auto TR_, auto FTV_) {
    fwd_loglik_kernel<N, VEC_, TR_, false, FTV_><<<g.blocks, kLlBlock, 0, stream>>>(
        md, a.y, a.T, g.M, w.X, tot, g.sub, part, last, 1, nullptr, a.Fd);
  }, inputs_aligned(a), o.transition != nullptr, a.Fd != nullptr);
  ++*launches;
  CK(cudaGetLastError());
  loglik_finish_kernel<<<1, kLlFinish, 0, stream>>>(part, g.blocks, last, N, o.transition, o.innovations,
                                                     o.m_last, o.C_last, o.status, nullptr);
  ++*launches;
  return cudaGetLastError();
}

// One rank's chunk of a time-sharded series after the all-gather of the forward aggregates: fold the
// carry (as the forward finish phase), sweep the chunk from it with both terms, and sum the block
// partials into the rank's [transition, innovations, status] vector o.part_vec.  X still holds the
// chunk's scanned prefixes from bdlm_scan_dist_forward_local.  The rank holding row T also writes
// (m_T, C_T) and flags a non-finite m_T in its status.
template <int N>
cudaError_t scan_dist_loglik(const ScanArgs &a, const ScanLoglikOut &o, cudaStream_t stream, int64_t *launches) {
  if (a.phase != kScanDistFinish) return cudaErrorInvalidValue;
  const ScanModel<N> md = make_model<N>(a);
  const ScanGeom g = scan_geom(a, kPassLoglik);
  const ScanLayout<FElem<N>> w(g, a.workspace);
  LoglikPart *part = reinterpret_cast<LoglikPart *>(o.parts);
  double *last = reinterpret_cast<double *>(part + g.blocks);
  const bool holds_last = a.rank == a.world - 1;
  fold_forward_kernel<N><<<1, 1, 0, stream>>>(reinterpret_cast<const FElem<N> *>(a.aggs_dev), a.rank,
                                              state_arg<N>(a.start), w.carry, ScanPeers{}, nullptr, nullptr);
  ++*launches;
  CK(cudaGetLastError());
  const FElem<N> *tot = g.nb > 1 ? w.scratch : nullptr;
  with_flags([&](auto VEC_, auto FTV_) {
    fwd_loglik_kernel<N, VEC_, true, true, FTV_><<<g.blocks, kLlBlock, 0, stream>>>(
        md, a.y, a.T, g.M, w.X, tot, g.sub, part, last, a.keep_init, w.carry, a.Fd);
  }, inputs_aligned(a), a.Fd != nullptr);
  ++*launches;
  CK(cudaGetLastError());
  loglik_finish_kernel<<<1, kLlFinish, 0, stream>>>(part, g.blocks, holds_last ? last : nullptr, N, o.part_vec,
                                                     o.part_vec + 1, o.m_last, o.C_last, nullptr, o.part_vec + 2);
  ++*launches;
  return cudaGetLastError();
}

template <int N>
bool sampler_vec(const ScanArgs &a, const ScanFfbsOut &o) {
  return dense_aligned(a.kf.m, N) && dense_aligned(a.kf.C, N * N) && dense_aligned(o.theta, N) &&
         inputs_aligned(a);
}

// The sampler's level 1 (elements, c_r into theta, the terminal slot) and its level-2 suffix scan.
// Rows 0 .. g.rows - 1 have a successor (all of them when another chunk follows); row g.rows is the
// series' last when no chunk follows (`terminal`).
template <int N>
cudaError_t sampler_prefixes(const ScanArgs &a, const ScanFfbsOut &o, const ScanGeom &g, cudaStream_t stream,
                             int64_t *launches) {
  const ScanModel<N> md = make_model<N>(a);
  const ScanLayout<BElem<N>> w(g, o.workspace);
  const FfbsRng rng{o.rng_seed, o.rng_sweep, o.rng_base, o.total_rows, o.first_row};
  const bool terminal = !a.has_successor;
  const int64_t term = terminal ? g.rows : -1;
  if (sampler_vec<N>(a, o))
    ffbs_reduce_kernel<N, true><<<g.blocks, kFbBlock, 0, stream>>>(md, a.kf.m, a.kf.C, g.rows, g.M, o.z, rng,
                                                                    o.theta, w.X, a.status, g.sub, term);
  else
    ffbs_reduce_kernel<N, false><<<g.blocks, kFbBlock, 0, stream>>>(md, a.kf.m, a.kf.C, g.rows, g.M, o.z, rng,
                                                                     o.theta, w.X, a.status, g.sub, term);
  ++*launches;
  CK(cudaGetLastError());
  // a chunk that others follow: the terminal slot is the identity, so its aggregate leaves the later
  // chunks to the carry; a last chunk of one row: its one thread folded no row
  if (!terminal || g.rows == 0) {
    set_b_identity<N><<<1, 1, 0, stream>>>(terminal ? w.X : w.X + g.M);
    ++*launches;
    CK(cudaGetLastError());
  }
  return device_scan<BElem<N>, true, true>(w.X, g.M + 1, w.scratch, stream, launches, /*defer_top=*/true);
}

// The apply sweep from the scanned suffixes (and the carry of later chunks), then, with statistics,
// the fixed-order sum of its block partials into `stats` or into the rank's partial vector `vec`.
template <int N>
cudaError_t sampler_apply(const ScanArgs &a, const ScanFfbsOut &o, const ScanGeom &g, const BElem<N> *carry,
                          bool stats, double *vec, cudaStream_t stream, int64_t *launches) {
  const ScanModel<N> md = make_model<N>(a);
  const ScanLayout<BElem<N>> w(g, o.workspace);
  const BElem<N> *tot = g.nb > 1 ? w.scratch : nullptr;
  const bool vec_io = sampler_vec<N>(a, o), terminal = !a.has_successor;
  // F enters the statistics only
  with_flags([&](auto VEC_, auto STATS_, auto FTV_) {
    ffbs_apply_kernel<N, VEC_, STATS_, FTV_ && STATS_><<<g.blocks, kFbBlock, 0, stream>>>(
        md, a.kf.m, a.kf.C, a.y, g.rows, g.M, w.X, tot, o.theta, a.status, g.sub, o.parts, carry, a.keep_init, a.T,
        terminal, a.Fd);
  }, vec_io, stats, a.Fd != nullptr);
  ++*launches;
  CK(cudaGetLastError());
  if (stats) {
    ffbs_stats_finish_kernel<N><<<1, kFbFinish, 0, stream>>>(o.parts, g.blocks, o.stats, vec, a.status);
    ++*launches;
  }
  return cudaGetLastError();
}

// FFBS of the whole series (keep_init = 1): the forward pass writes (m, C) (+ whatever of a, R, f, Q
// a.kf asks for), then the sampler's level 1, its level-2 suffix scan, the apply sweep and, with
// statistics, the fixed-order sum of the apply's block partials.
template <int N>
cudaError_t scan_ffbs(const ScanArgs &a, const ScanFfbsOut &o, cudaStream_t stream, int64_t *launches) {
  if (a.keep_init != 1 || a.phase != kScanApply || a.fuse_sagg || a.has_successor) return cudaErrorInvalidValue;
  CK(scan_forward<N>(a, stream, launches));
  const ScanGeom g = scan_geom(a, kPassSampler);
  CK(sampler_prefixes<N>(a, o, g, stream, launches));
  const StatViews &sv = o.stats;
  const bool stats = sv.ssy.ptr || sv.ny.ptr || sv.ssw.ptr || sv.scatter.ptr;
  return sampler_apply<N>(a, o, g, nullptr, stats, nullptr, stream, launches);
}

// One rank's chunk of a time-sharded FFBS.  Local (a.phase = kScanDistFinish of the forward pass): the
// forward finish with (m, C) into a.kf and no smoother fold, then the sampler's level 1 + level 2 and
// the chunk's aggregate into o.agg_dev for the all-gather.  Finish: fold the carry of the later
// chunks from o.aggs_dev, apply, and sum the statistics and status into the partial vector o.part_vec.
template <int N>
cudaError_t scan_dist_ffbs(const ScanArgs &a, const ScanFfbsOut &o, bool finish, cudaStream_t stream,
                           int64_t *launches) {
  if (a.phase != kScanDistFinish || a.fuse_sagg) return cudaErrorInvalidValue;
  const ScanGeom g = scan_geom(a, kPassSampler);
  const ScanLayout<BElem<N>> w(g, o.workspace);
  if (!finish) {
    CK(scan_forward<N>(a, stream, launches));
    CK(sampler_prefixes<N>(a, o, g, stream, launches));
    const BElem<N> *whole = g.nb > 1 ? w.scratch + (g.nb - 1) : w.X;  // suffix scan ends at index 0
    return cudaMemcpyAsync(o.agg_dev, whole, sizeof(BElem<N>), cudaMemcpyDeviceToDevice, stream);
  }
  if (a.has_successor) {
    fold_sampler_kernel<N><<<1, 1, 0, stream>>>(reinterpret_cast<const BElem<N> *>(o.aggs_dev), a.rank, a.world,
                                                w.carry);
    ++*launches;
    CK(cudaGetLastError());
  }
  return sampler_apply<N>(a, o, g, a.has_successor ? w.carry : nullptr, true, o.part_vec, stream, launches);
}

template <int N>
cudaError_t scan_backward(const ScanArgs &a, cudaStream_t stream, int64_t *launches) {
  const ScanModel<N> md = make_model<N>(a);
  // rows with a successor inside this chunk: all but the last, plus the last when the chunk
  // is followed by another one (has_successor)
  const ScanGeom g = scan_geom(a, kPassBackward);
  const ScanLayout<SElem<N>> w(g, a.workspace);
  const bool local = a.phase == kScanDistLocal, finish = a.phase == kScanDistFinish;
  const bool vec = dense_aligned(a.kf.m, N) && dense_aligned(a.kf.C, N * N) &&
                   dense_aligned(a.s, N) && dense_aligned(a.S, N * N);
  if (!finish) {
    // X[0, M) already holds the level-1 aggregates, written by the forward apply sweep (fuse_sagg)
    if (a.has_successor) {  // dist local of a chunk followed by others
      set_s_identity<N><<<1, 1, 0, stream>>>(w.X + g.M);
    } else {  // last chunk: s_T = m_T, S_T = C_T at its last row, g.rows (Smoothing.scala:59-61)
      terminal_from_last_row<N><<<1, 1, 0, stream>>>(a.kf.m, a.kf.C, g.rows, a.s, a.S, w.X + g.M,
                                                     g.M == 0 ? a.status : nullptr);
    }
    ++*launches;
    CK(cudaGetLastError());
    CK((device_scan<SElem<N>, true, true>(w.X, g.M + 1, w.scratch, stream, launches, /*defer_top=*/true)));
    const SElem<N> *whole = g.nb > 1 ? w.scratch + (g.nb - 1) : w.X;  // the whole chunk (suffix scan ends at index 0)
    if (local) {
      if (a.peers.world > 0) {
        publish_kernel<SElem<N>><<<a.peers.world, 64, 0, stream>>>(whole, a.peers, a.rank, a.epoch_dev);
        ++*launches;
        return cudaGetLastError();
      }
      return cudaMemcpyAsync(a.agg_dev, whole, sizeof(SElem<N>), cudaMemcpyDeviceToDevice, stream);
    }
  } else if (a.has_successor) {
    fold_backward_kernel<N><<<1, 1, 0, stream>>>(reinterpret_cast<const SElem<N> *>(a.aggs_dev),
                                                 a.rank, a.world, w.carry, a.peers, a.epoch_dev, a.status);
    ++*launches;
  }
  const SElem<N> *cr = (finish && a.has_successor) ? w.carry : nullptr;
  const SElem<N> *tot = g.nb > 1 ? w.scratch : nullptr;
  if (g.M > 0) {
    if (vec)
      bwd_apply_kernel<N, true><<<g.blocks, 128, 0, stream>>>(md, a.kf.m, a.kf.C, g.rows, g.M, w.X, a.s, a.S,
                                                              a.status, cr, tot, g.sub);
    else
      bwd_apply_kernel<N, false><<<g.blocks, 128, 0, stream>>>(md, a.kf.m, a.kf.C, g.rows, g.M, w.X, a.s, a.S,
                                                               a.status, cr, tot, g.sub);
    ++*launches;
  }
  return cudaGetLastError();
}

}  // namespace

// Every pass over a chunk of T observations fits the forward pass's layout with keep_init = 1: no
// pass has more level-1 threads, and no element is larger than the forward one.
size_t scan_workspace_bytes(int n, int64_t T) {
  const ScanGeom g = scan_geom(n, T, 1, false, kPassForward);
  return with_n(n, (size_t)0, [&](auto N) { return ScanLayout<FElem<N>>::bytes(g); });
}

__global__ void epoch_bump_kernel(unsigned long long *epoch_dev) { *epoch_dev = *epoch_dev + 1; }
cudaError_t launch_epoch_bump(unsigned long long *epoch_dev, cudaStream_t stream) {
  epoch_bump_kernel<<<1, 1, 0, stream>>>(epoch_dev);
  return cudaGetLastError();
}

size_t scan_table_bytes() { return kScanTableBytes; }
int scan_forward_elem_doubles(int n) { return 3 * n * n + 2 * n; }
int scan_backward_elem_doubles(int n) { return 2 * n * n + n; }

cudaError_t launch_scan(const ScanArgs &a, cudaStream_t stream, int64_t *launches) {
  return with_n(a.n, cudaErrorInvalidValue, [&](auto N) {
    return a.backward ? scan_backward<N>(a, stream, launches) : scan_forward<N>(a, stream, launches);
  });
}

// block partials, then the last state (n + n*n doubles); a chunk with keep_init = 0 has no more blocks
size_t scan_loglik_bytes(int n, int64_t T) {
  return sizeof(LoglikPart) * (size_t)scan_geom(n, T, 1, false, kPassLoglik).blocks +
         sizeof(double) * (size_t)(n + n * n);
}

cudaError_t launch_scan_loglik(const ScanArgs &a, const ScanLoglikOut &o, cudaStream_t stream,
                               int64_t *launches) {
  return with_n(a.n, cudaErrorInvalidValue, [&](auto N) { return scan_loglik<N>(a, o, stream, launches); });
}

// 2 + n + n*n statistics per block of the sampler's sweep over any chunk of T observations
size_t scan_ffbs_parts_bytes(int n, int64_t T) {
  return sizeof(double) * (size_t)(2 + n + n * n) * (size_t)scan_geom(n, T, 1, true, kPassSampler).blocks;
}

cudaError_t launch_scan_ffbs(const ScanArgs &a, const ScanFfbsOut &o, cudaStream_t stream, int64_t *launches) {
  return with_n(a.n, cudaErrorInvalidValue, [&](auto N) { return scan_ffbs<N>(a, o, stream, launches); });
}

cudaError_t launch_scan_dist_loglik(const ScanArgs &a, const ScanLoglikOut &o, cudaStream_t stream,
                                    int64_t *launches) {
  return with_n(a.n, cudaErrorInvalidValue, [&](auto N) { return scan_dist_loglik<N>(a, o, stream, launches); });
}

cudaError_t launch_scan_dist_loglik_finish(const double *parts, int world, double *transition, double *innovations,
                                           int32_t *status, cudaStream_t stream, int64_t *launches) {
  dist_loglik_finish_kernel<<<1, 1, 0, stream>>>(parts, world, transition, innovations, status);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_scan_dist_ffbs(const ScanArgs &a, const ScanFfbsOut &o, bool finish, cudaStream_t stream,
                                  int64_t *launches) {
  return with_n(a.n, cudaErrorInvalidValue,
                [&](auto N) { return scan_dist_ffbs<N>(a, o, finish, stream, launches); });
}

cudaError_t launch_scan_dist_ffbs_stats_finish(int n, const double *parts, int world, const StatViews &sv,
                                               int32_t *status, cudaStream_t stream, int64_t *launches) {
  return with_n(n, cudaErrorInvalidValue, [&](auto N) {
    dist_ffbs_stats_finish_kernel<N><<<1, 1, 0, stream>>>(parts, world, sv, status);
    ++*launches;
    return cudaGetLastError();
  });
}

int scan_sampler_elem_doubles(int n) { return n * n + n; }

// Host build of the combine the kernels inline: out = ei (x) ej (ei earlier in time).
void scan_combine_host(int n, bool backward, const double *ei, const double *ej, double *out) {
  with_n(n, 0, [&](auto N) {
    if (backward)
      s_combine<N>(*reinterpret_cast<const SElem<N> *>(ei), *reinterpret_cast<const SElem<N> *>(ej),
                   *reinterpret_cast<SElem<N> *>(out));
    else
      f_combine<N>(*reinterpret_cast<const FElem<N> *>(ei), *reinterpret_cast<const FElem<N> *>(ej),
                   *reinterpret_cast<FElem<N> *>(out));
    return 0;
  });
}

}  // namespace bdlm
