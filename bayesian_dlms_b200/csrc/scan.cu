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
//
// Multi-GPU: a rank's chunk aggregate (3n^2+2n doubles forward, 2n^2+n backward) is all
// that crosses the fabric (one all-gather per pass); the carry is folded on the host.
//
// Parity: equals the sequential kernel in textbook-smoother mode to 1e-9 relative (for n = 1
// that is the reference itself); the apply phases reuse the sequential step code, so the
// only difference is the rounding of the scanned start states.
#include <cmath>
#include <vector>

#include "common.cuh"
#include "launch.h"
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

template <int N, bool VEC>
__global__ void __launch_bounds__(128)
fwd_reduce_kernel(const ScanModel<N> md, const FwdTable<N> *__restrict__ tb,
                  const double *__restrict__ y, int64_t T, int64_t M, int keep_init,
                  FElem<N> *agg /* [M + 1], slot 0 = the start element */,
                  const StateArg<N> start, bool identity_start, int sub) {
  const int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (c >= M) return;
  if (c == 0) {  // slot 0: the state before the chunk, or the identity (aggregate-only phases)
    FElem<N> e0;
    if (identity_start) f_identity<N>(e0); else f_state<N>(e0, start.v, start.v + N);
    agg[0] = e0;
  }
  const int64_t rows = T + keep_init;
  const int64_t r0 = c * (int64_t)sub, r1 = (r0 + sub < rows) ? r0 + sub : rows;
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
__device__ __forceinline__ void fwd_row(const ScanModel<N> &md, const double (&W)[N * N], bool init_row,
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
    update<N, true>(md.F, md.V, yv, o.a, o.R, o.f, o.Q, m, C, st);
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

// The two apply sweeps ask ptxas for one resident block per SM: asking for more makes them spill,
// which costs more than the occupancy gains (profiles/r1_tuning.txt, "scan apply sweeps").
template <int N, bool VEC, bool FUSE>
__global__ void __launch_bounds__(128, 1)
fwd_apply_kernel(const ScanModel<N> md, const double *__restrict__ y, int64_t T, int64_t M,
                 const FElem<N> *pre /* [M+1] inclusive scan with slot 0 = start */,
                 int keep_init, KfViews kf, int32_t *status,
                 SElem<N> *sagg /* FUSE: smoother level-1 aggregates */, int64_t nrows,
                 const FElem<N> *carry /* multi-GPU: everything before this chunk, or nullptr */,
                 const FElem<N> *tot /* scanned level-2 block totals whose prefix `pre` still lacks, or nullptr */,
                 int sub) {
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
    yg.start(y, r0, keep_init);
    for (; r + kGrp <= r1; r += kGrp) {
      double yv[kGrp];
      yg.load(y, r, T, keep_init, yv);
      GroupBuf<N> ga, gm;
      GroupBuf<N * N> gR, gC;
      GroupBuf<1> gf, gQ;
#define BDLM_FWD_ROW(I)                                                          \
  {                                                                              \
    FwdRow<N> o;                                                                 \
    fwd_row<N, FUSE>(md, W, keep_init && r + I == 0, yv[I], m, C, an, Rn, o, st, \
                     r + I < nrows, sacc, shave);                                \
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
    fwd_row<N, FUSE>(md, W, t < 0, t >= 0 ? y[t] : 0.0, m, C, an, Rn, o, st, r < nrows, sacc, shave);
    store_row_scalar<N>(kf.a, r, o.a); store_row_scalar<N * N>(kf.R, r, o.R);
    store_row_scalar<1>(kf.f, r, &o.f); store_row_scalar<1>(kf.Q, r, &o.Q);
    store_row_scalar<N>(kf.m, r, o.m); store_row_scalar<N * N>(kf.C, r, o.C);
  }
  if (FUSE && shave) sagg[c] = sacc;
  if (status && st) atomicOr(status, st);
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

// terminal slot of a chunk that others follow: the identity, so that the chunk's aggregate leaves
// them out (the finish phase brings them in through the carry)
template <int N>
__global__ void set_s_identity(SElem<N> *slot) {
  SElem<N> e;
  s_identity<N>(e);
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

int scan_rows_per_thread(int n, int64_t T) {
  int slots = 444;
  switch (n) {
    case 1: slots = apply_slots<1>(); break;
    case 2: slots = apply_slots<2>(); break;
    case 3: slots = apply_slots<3>(); break;
    case 4: slots = apply_slots<4>(); break;
    default: break;
  }
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

template <int N>
ScanModel<N> make_model(const ScanArgs &a) {
  ScanModel<N> md;
  for (int k = 0; k < N * N; ++k) { md.G[k] = a.G[k]; md.W[k] = a.W[k]; }
  for (int k = 0; k < N; ++k) md.F[k] = a.F[k];
  md.V = a.V;
  return md;
}

#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return e_; } while (0)

// 256-bit path: dense rows (sk = 1, sr = K) on a 32-byte aligned base.
static bool dense_aligned(const View &v, int64_t K) {
  return !v.ptr || (v.sk == 1 && v.sr == K && (reinterpret_cast<uintptr_t>(v.ptr) & 31) == 0);
}

template <int N>
cudaError_t scan_forward(const ScanArgs &a, cudaStream_t stream, int64_t *launches) {
  const ScanModel<N> md = make_model<N>(a);
  const int sub = scan_rows_per_thread(a.n, a.T);
  const int64_t T = a.T, M = (T + a.keep_init + sub - 1) / sub;
  FElem<N> *X = reinterpret_cast<FElem<N> *>(a.workspace);       // [M + 1]
  FElem<N> *scratch = X + (M + 1);                                // block totals
  const unsigned blocks = (unsigned)((M + 127) / 128);
  const int64_t nb = (M + 1 + kScanBlock * kPer - 1) / (kScanBlock * kPer);  // level-2 blocks over X
  FwdTable<N> *tb = reinterpret_cast<FwdTable<N> *>(a.table);
  if (a.table_upload) {  // model changed since the context last built it
    static_assert(sizeof(FwdTable<N>) <= kScanTableBytes, "table buffer too small");
    FwdTable<N> host;
    build_fwd_table<N>(md, host);
    // pageable source: staged by the driver before the call returns
    CK(cudaMemcpyAsync(tb, &host, sizeof(host), cudaMemcpyHostToDevice, stream));
  }
  const bool local = a.phase == kScanDistLocal, finish = a.phase == kScanDistFinish;
  FElem<N> *carry = reinterpret_cast<FElem<N> *>(scratch + (M + 1) / kScanBlock * 2 + 8);
  if (!finish) {
    // dist local: chunk aggregate only (identity start); apply: prefix of
    // (start (x) aggregates), a.start = host (m, C) of the state before t = 0
    const StateArg<N> st0 = state_arg<N>(local ? nullptr : a.start);
    if ((reinterpret_cast<uintptr_t>(a.y) & 31) == 0)
      fwd_reduce_kernel<N, true><<<blocks, 128, 0, stream>>>(md, tb, a.y, T, M, a.keep_init, X, st0, local, sub);
    else
      fwd_reduce_kernel<N, false><<<blocks, 128, 0, stream>>>(md, tb, a.y, T, M, a.keep_init, X, st0, local, sub);
    ++*launches;
    CK(cudaGetLastError());
    CK((device_scan<FElem<N>, false, false>(X, M + 1, scratch, stream, launches, /*defer_top=*/true)));
    // the whole chunk: last element of a one-block scan, else the last scanned block total
    const FElem<N> *whole = nb > 1 ? scratch + (nb - 1) : X + M;
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
                                                a.rank, state_arg<N>(a.start), carry, a.peers,
                                                a.epoch_dev, a.status);
    ++*launches;
  }
  const bool vec = dense_aligned(a.kf.m, N) && dense_aligned(a.kf.C, N * N) &&
                   dense_aligned(a.kf.a, N) && dense_aligned(a.kf.R, N * N) &&
                   dense_aligned(a.kf.f, 1) && dense_aligned(a.kf.Q, 1) &&
                   (reinterpret_cast<uintptr_t>(a.y) & 31) == 0;
  // a.fuse_sagg: the caller runs the smoother next on the same rows: fold the smoothing
  // elements here so the backward pass starts from ready level-1 aggregates.
  SElem<N> *sagg = reinterpret_cast<SElem<N> *>(a.fuse_sagg);
  const int64_t nrows = T + a.keep_init - (a.has_successor ? 0 : 1);
  const FElem<N> *cr = finish ? carry : nullptr;
  const FElem<N> *tot = nb > 1 ? scratch : nullptr;  // top-level block prefixes, composed by the sweep
#define BDLM_FWD_APPLY(VEC_, FUSE_)                                                         \
  fwd_apply_kernel<N, VEC_, FUSE_><<<blocks, 128, 0, stream>>>(md, a.y, T, M, X, a.keep_init, \
                                                               a.kf, a.status, sagg, nrows, cr, tot, sub)
  if (vec && sagg) BDLM_FWD_APPLY(true, true);
  else if (vec) BDLM_FWD_APPLY(true, false);
  else if (sagg) BDLM_FWD_APPLY(false, true);
  else BDLM_FWD_APPLY(false, false);
#undef BDLM_FWD_APPLY
  ++*launches;
  return cudaGetLastError();
}

template <int N>
cudaError_t scan_backward(const ScanArgs &a, cudaStream_t stream, int64_t *launches) {
  const ScanModel<N> md = make_model<N>(a);
  const int64_t rows = a.T + a.keep_init;
  // rows with a successor inside this chunk: all but the last, plus the last when the chunk
  // is followed by another one (has_successor)
  const int64_t nrows = a.has_successor ? rows : rows - 1;
  const int sub = scan_rows_per_thread(a.n, a.T);
  const int64_t M = (nrows + sub - 1) / sub;
  SElem<N> *X = reinterpret_cast<SElem<N> *>(a.workspace);  // [M + 1]
  SElem<N> *scratch = X + (M + 1);
  double *term_dev = reinterpret_cast<double *>(scratch + (M + 1) / kScanBlock * 2 + 8);
  const unsigned blocks = (unsigned)((M + 127) / 128);
  const int64_t nb = (M + 1 + kScanBlock * kPer - 1) / (kScanBlock * kPer);  // level-2 blocks over X
  const bool local = a.phase == kScanDistLocal, finish = a.phase == kScanDistFinish;
  const bool vec = dense_aligned(a.kf.m, N) && dense_aligned(a.kf.C, N * N) &&
                   dense_aligned(a.s, N) && dense_aligned(a.S, N * N);
  SElem<N> *carry = reinterpret_cast<SElem<N> *>(term_dev + 64);
  if (!finish) {
    // X[0, M) already holds the level-1 aggregates, written by the forward apply sweep (fuse_sagg)
    if (a.has_successor) {  // dist local of a chunk followed by others
      set_s_identity<N><<<1, 1, 0, stream>>>(X + M);
    } else {  // last chunk: s_T = m_T, S_T = C_T (Smoothing.scala:59-61)
      terminal_from_last_row<N><<<1, 1, 0, stream>>>(a.kf.m, a.kf.C, rows - 1, a.s, a.S, X + M,
                                                     M == 0 ? a.status : nullptr);
    }
    ++*launches;
    CK(cudaGetLastError());
    CK((device_scan<SElem<N>, true, true>(X, M + 1, scratch, stream, launches, /*defer_top=*/true)));
    const SElem<N> *whole = nb > 1 ? scratch + (nb - 1) : X;  // the whole chunk (suffix scan ends at index 0)
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
                                                 a.rank, a.world, carry, a.peers, a.epoch_dev, a.status);
    ++*launches;
  }
  const SElem<N> *cr = (finish && a.has_successor) ? carry : nullptr;
  const SElem<N> *tot = nb > 1 ? scratch : nullptr;
  if (M > 0) {
    if (vec)
      bwd_apply_kernel<N, true><<<blocks, 128, 0, stream>>>(md, a.kf.m, a.kf.C, nrows, M, X, a.s, a.S, a.status, cr, tot, sub);
    else
      bwd_apply_kernel<N, false><<<blocks, 128, 0, stream>>>(md, a.kf.m, a.kf.C, nrows, M, X, a.s, a.S, a.status, cr, tot, sub);
    ++*launches;
  }
  return cudaGetLastError();
}

}  // namespace

size_t scan_workspace_bytes(int n, int64_t T) {
  const int sub = scan_rows_per_thread(n, T);
  const int64_t M = (T + 1 + sub - 1) / sub + 2;
  const size_t elem = sizeof(double) * (3 * n * n + 2 * n);
  return elem * (size_t)(M + 1 + (M + 1) / kScanBlock * 2 + 24) + 8192;
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
  switch (a.n) {
#define BDLM_SCAN_CASE(N_)                                                         \
  case N_:                                                                         \
    return a.backward ? scan_backward<N_>(a, stream, launches) : scan_forward<N_>(a, stream, launches);
    BDLM_SCAN_CASE(1)
    BDLM_SCAN_CASE(2)
    BDLM_SCAN_CASE(3)
    BDLM_SCAN_CASE(4)
#undef BDLM_SCAN_CASE
    default: return cudaErrorInvalidValue;
  }
}

// Host build of the combine the kernels inline: out = ei (x) ej (ei earlier in time).
void scan_combine_host(int n, bool backward, const double *ei, const double *ej, double *out) {
  switch (n) {
#define BDLM_COMB_CASE(N_)                                                                  \
  case N_:                                                                                  \
    if (backward) s_combine<N_>(*reinterpret_cast<const SElem<N_> *>(ei),                   \
                                *reinterpret_cast<const SElem<N_> *>(ej),                   \
                                *reinterpret_cast<SElem<N_> *>(out));                       \
    else f_combine<N_>(*reinterpret_cast<const FElem<N_> *>(ei),                            \
                       *reinterpret_cast<const FElem<N_> *>(ej),                            \
                       *reinterpret_cast<FElem<N_> *>(out));                                \
    break;
    BDLM_COMB_CASE(1)
    BDLM_COMB_CASE(2)
    BDLM_COMB_CASE(3)
    BDLM_COMB_CASE(4)
#undef BDLM_COMB_CASE
    default: break;
  }
}

}  // namespace bdlm
