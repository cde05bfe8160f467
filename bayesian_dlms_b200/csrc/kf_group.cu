// kf_group.cu -- FFBS / filter for mid-size state dimension, p = 1 (BASELINE config 3:
// polynomial(1) |+| seasonal(24, 6), n = 13): SIXTEEN LANES PER SERIES, TWO SERIES PER WARP,
// compile-time n.
//
// These shapes are FP64-issue bound (about 180 kflop against 3 KB per FFBS step), and most of
// the work is the Jacobi eigen-decomposition behind MultivariateGaussianSvd.draw.  Compared
// with the generic warp-per-series kernel (kf_warp.cu) this kernel
//   * packs two series into every warp-instruction (13 of 16 lanes busy instead of 13 of 32),
//   * gives lane j COLUMN j of every matrix in registers, with all loops unrolled at compile
//     time (static register indexing, no index arithmetic); products are always
//     (matrix in shared memory, read by broadcast) x (column in registers),
//   * runs the round-robin Jacobi schedule with lane j owning column j of A and V: per round a
//     lane reads its partner's column from shared memory and applies the fused two-sided
//     rotation to its own column (rounds are a run-time loop: unrolling them made the kernel
//     466 KB of code and ncu showed 87 % "no instruction" stalls, see profiles/).
// Every output element is still produced by one lane with the oracle's operation order, so
// results stay bit-identical to oracle/bdlm_oracle.c (asserted by tests/test_gpu_parity.py).
//
// Reference: Smoothing.ffbs / sample / step (Smoothing.scala:74-159), KalmanFilter.step
// (KalmanFilter.scala:64-107,273-321), MultivariateGaussianSvd.draw (:13-22), Gibbs
// sufficient statistics (Gibbs.scala:29-43,63-73; GibbsWishart.scala:22-29).
#include "common.cuh"
#include "launch.h"
#include "rng.cuh"
#include "warp_linalg.cuh"

namespace bdlm {
namespace {

constexpr int GW = 16;      // lanes per series
constexpr int kWpb = 2;     // warps per block

template <int N>
struct GSmem {               // per SERIES shared memory (doubles)
  static constexpr int LD = N | 1;  // odd leading dimension: column reads by 16 lanes hit 16 banks
  static constexpr int MAT = LD * N;
  static constexpr int VEC = 16;
  static constexpr int kMats = 4;   // S0..S3 per series (W is read from global / L1 where it is
                                    // used: one column per lane per step; G: one copy per WARP)
  static constexpr int kVecs = 6;
  static constexpr int total = kMats * MAT + kVecs * VEC;   // per series
  static constexpr int warp_total = 2 * total + MAT;        // two series + the shared model G
};

// out[i] = sum_k X[i + k*LD] * y[k]   (X in shared memory, broadcast reads)
template <int N, int LD>
__device__ __forceinline__ void mm_sx(const double *X, const double (&y)[N], double (&out)[N]) {
#pragma unroll
  for (int i = 0; i < N; ++i) {
    double acc = 0.0;
#pragma unroll
    for (int k = 0; k < N; ++k) {
      const double prod = X[i + k * LD] * y[k];
      acc = (k == 0) ? prod : acc + prod;
    }
    out[i] = acc;
  }
}

// out[i] = sum_k X[i + k*LD] * y[k*ys] with the k loop at RUN time (rows i stay compile-time
// register indices): the same products summed in the same order as mm_sx, in 1/12 of the code.
// The straight-line body of an FFBS step was 150 KB of SASS that every warp streamed once per
// step (ncu: 2.7 warps per issue-active cycle stalled on instruction fetch,
// profiles/r2_group_onesided_full.txt); y comes from shared memory (or, for W, global memory).
template <int N, int LD>
__device__ __forceinline__ void mm_sy(const double *X, const double *y, int64_t ys, double (&out)[N]) {
  {
    const double y0 = y[0];
#pragma unroll
    for (int i = 0; i < N; ++i) out[i] = X[i] * y0;
  }
#pragma unroll 1
  for (int k = 1; k < N; ++k) {
    const double yk = y[k * ys];
    const double *xc = X + k * LD;
#pragma unroll
    for (int i = 0; i < N; ++i) out[i] = out[i] + xc[i] * yk;
  }
}

template <int N>
struct Ctx {
  int lane, gl, grp;       // lane in warp, lane in group, group in warp
  bool act;                // gl < N
  int jj;                  // min(gl, N-1): safe index for addressing
  double *S0, *S1, *S2, *S3, *SG;
  double *VA, *VB, *VD, *VK, *VZ, *VX;
};

// ---- eigSym (oracle jacobi_eigsym) on REGISTER columns --------------------------------------
// One-sided Jacobi: lane j owns column j of U (= A at the start) and of V for the whole
// decomposition.  Per round a lane fetches its partner's U column by width-16 shuffles, forms
// |own|^2 and own . partner (the partner's norm arrives by one more shuffle: it sums the same
// squares in the same order, so alpha / beta / gamma are the oracle's bits in both lanes of the
// pair), derives (c, s) and rotates its own U and V columns:  own' = c * own + s' * partner with
// s' = -s in the lower-index lane (c*up - s*uq) and +s in the higher one (s*up + c*uq).  Nothing
// lives in shared memory, there is no barrier inside a sweep, no dependence on the OTHER pairs'
// rotation parameters and no lower / upper-triangle case split: about 300 instructions per round
// against 1000 for the two-sided update J^T A J this kernel used in round 1 (ncu, n = 13: 83 k
// instructions per FFBS step, 21 % of them FP64; profiles/r2_group_twosided_full.txt).
template <int N>
__device__ __forceinline__ bool jacobi_round(const Ctx<N> &cx, int round, double (&u)[N],
                                             double (&v)[N]) {
  const int j = cx.jj;
  const int q = cx.act ? rr_partner(N, round, j) : -1;
  const int src = q < 0 ? cx.gl : q;   // lane (in the 16-lane group) holding the partner column
  const bool low = j < q;
  double w[N];
  double own = 0.0, gamma = 0.0;
#pragma unroll
  for (int i = 0; i < N; ++i) {
    w[i] = __shfl_sync(FULL, u[i], src, GW);
    const double sq = u[i] * u[i], pq = u[i] * w[i];
    own = (i == 0) ? sq : own + sq;
    gamma = (i == 0) ? pq : gamma + pq;
  }
  const double other = __shfl_sync(FULL, own, src, GW);
  const double alpha = low ? own : other, beta = low ? other : own;
  const bool rot = q >= 0 && (gamma * gamma > kJacobiThr2 * (alpha * beta));
  // nobody in the warp rotates (the last sweep of both series): skip the V exchange as well
  if (__ballot_sync(FULL, rot) == 0u) return false;
  double c = 1.0, sp = 0.0;
  if (rot) {
    double cc, ss;
    sym_rot(alpha, beta, gamma, cc, ss);
    c = cc;
    sp = low ? -ss : ss;
  }
#pragma unroll
  for (int i = 0; i < N; ++i) {
    const double vw = __shfl_sync(FULL, v[i], src, GW);
    if (rot) {
      u[i] = c * u[i] + sp * w[i];
      v[i] = c * v[i] + sp * vw;
    }
  }
  return rot;
}

// MultivariateGaussianSvd(mu, cov).draw with injected normals.  Input: the symmetric matrix
// whose LOWER triangle is read sits in S0 (column-major, ld LD); mu_j, z_j per lane.
// Uses S3 (M = V diag(sqrt lam)), VL, VZ.  Returns the draw element of lane j.
template <int N>
__device__ __noinline__ double eig_draw(const Ctx<N> cx, double mu_j, double z_j, int &st) {
  constexpr int LD = GSmem<N>::LD;
  const int j = cx.jj;
  double u[N], v[N];
#pragma unroll
  for (int i = 0; i < N; ++i) {
    u[i] = (i >= j) ? cx.S0[i + j * LD] : cx.S0[j + i * LD];
    v[i] = (i == j) ? 1.0 : 0.0;
  }
  if (cx.act) cx.VZ[j] = z_j;
  constexpr int M = (N + 1) & ~1;
  bool converged_grp = (N == 1);
  const unsigned gbits = 0xffffu << (cx.grp * GW);
  for (int sweep = 0; sweep < kJacobiMaxSweeps && N > 1; ++sweep) {
    bool rot = false;
    for (int round = 0; round < M - 1; ++round) rot = jacobi_round<N>(cx, round, u, v) || rot;
    const unsigned bal = __ballot_sync(FULL, rot);
    if ((bal & gbits) == 0u) converged_grp = true;  // this series saw a sweep without a rotation
    // continue while either series of the warp still rotates (a converged series only executes
    // no-op rounds, exactly like the oracle's `continue`)
    if (bal == 0u) break;
  }
  if (!converged_grp) st |= BDLM_ST_NOTCONVERGED;
  // lam_j = sign(v_j . u_j) |u_j|; ascending (stable), sign rule, M = V diag(sqrt lam) sorted
  double nn = 0.0, dot = 0.0;
#pragma unroll
  for (int i = 0; i < N; ++i) {
    const double sq = u[i] * u[i], vu = v[i] * u[i];
    nn = (i == 0) ? sq : nn + sq;
    dot = (i == 0) ? vu : dot + vu;
  }
  const double nrm = sqrt(nn);
  const double lam = (dot < 0.0) ? -nrm : nrm;
  int rank = 0;
#pragma unroll
  for (int k = 0; k < N; ++k) {
    const double lk = __shfl_sync(FULL, lam, k, GW);
    rank += ((lk < lam) || (lk == lam && k < j)) ? 1 : 0;
  }
  int im = 0;
  double best = fabs(v[0]);
#pragma unroll
  for (int i = 1; i < N; ++i) {
    const double a = fabs(v[i]);
    if (a > best) { best = a; im = i; }
  }
  double vim = v[0];
#pragma unroll
  for (int i = 1; i < N; ++i) vim = (im == i) ? v[i] : vim;
  const bool flip = vim < 0.0;
  const double sq = sqrt(lam);
  if (cx.act) {
#pragma unroll
    for (int i = 0; i < N; ++i) {
      const double x = flip ? -v[i] : v[i];
      cx.S3[i + rank * LD] = x * sq;
    }
  }
  __syncwarp();
  double x = 0.0;
#pragma unroll
  for (int k = 0; k < N; ++k) {
    const double prod = cx.S3[j + k * LD] * cx.VZ[k];
    x = (k == 0) ? prod : x + prod;
  }
  __syncwarp();
  return mu_j + x;
}

// dgesv restatement, column-distributed: lane j holds column j of A (N) and column j of the
// right-hand side (N); returns X column j in `rhs`.  Uses S2 for the factored matrix.
template <int N>
__device__ __forceinline__ int lu_cols(const Ctx<N> &cx, double (&A)[N], double (&rhs)[N]) {
  constexpr int LD = GSmem<N>::LD;
  const int j = cx.jj;
  const int base = cx.grp * GW;
  int st = 0;
#pragma unroll
  for (int j0 = 0; j0 < N; ++j0) {
    // pivot search in column j0 (held by lane j0)
    int jp_l = j0;
    double best = fabs(A[j0]);
#pragma unroll
    for (int i = j0 + 1; i < N; ++i) {
      const double v = fabs(A[i]);
      if (v > best) { best = v; jp_l = i; }
    }
    double pv_l = A[j0];
#pragma unroll
    for (int i = j0 + 1; i < N; ++i) pv_l = (jp_l == i) ? A[i] : pv_l;
    const int jp = __shfl_sync(FULL, jp_l, base + j0);
    const double pv = __shfl_sync(FULL, pv_l, base + j0);
    if (pv != 0.0) {
#pragma unroll
      for (int i = j0 + 1; i < N; ++i)
        if (jp == i) {
          double t = A[j0]; A[j0] = A[i]; A[i] = t;
          t = rhs[j0]; rhs[j0] = rhs[i]; rhs[i] = t;
        }
      const double r = 1.0 / A[j0];
      if (cx.gl == j0) {
#pragma unroll
        for (int i = j0 + 1; i < N; ++i) A[i] = A[i] * r;
      }
    } else {
      st = BDLM_ST_SINGULAR;
    }
#pragma unroll
    for (int i = j0 + 1; i < N; ++i) {
      const double l = __shfl_sync(FULL, A[i], base + j0);
      if (cx.gl > j0) A[i] = A[i] - l * A[j0];
      rhs[i] = rhs[i] - rhs[j0] * l;
    }
  }
  // publish U (upper triangle incl. diagonal) and back-substitute my right-hand side
  __syncwarp();
  if (cx.act) {
#pragma unroll
    for (int i = 0; i < N; ++i) cx.S2[i + j * LD] = A[i];
  }
  __syncwarp();
#pragma unroll
  for (int k = N - 1; k >= 0; --k) {
    rhs[k] = rhs[k] / cx.S2[k + k * LD];
#pragma unroll
    for (int i = 0; i < k; ++i) rhs[i] = rhs[i] - rhs[k] * cx.S2[i + k * LD];
  }
  __syncwarp();
  return st;
}

// 14 warps per SM (7 blocks): 148 x 14 x 2 = 4144 chains resident, so BASELINE config 3 (4096
// chains) is ONE wave; ptxas gets 65536 / (14 x 32) = 146 registers per thread.
template <int N, int OP>
__global__ void __launch_bounds__(kWpb * 32, 7)
group_kernel(const WarpArgs wa) {
  extern __shared__ double smem[];
  constexpr int LD = GSmem<N>::LD, MAT = GSmem<N>::MAT, VEC = GSmem<N>::VEC, NN = N * N;
  const Batch &bt = wa.bt;
  Ctx<N> cx;
  cx.lane = threadIdx.x & 31;
  cx.gl = cx.lane & (GW - 1);
  cx.grp = cx.lane >> 4;
  cx.act = cx.gl < N;
  cx.jj = cx.act ? cx.gl : N - 1;
  const int wib = threadIdx.x >> 5;
  const int sib = wib * 2 + cx.grp;  // series in block
  // the last series of an odd batch is processed twice (second copy writes nothing)
  int64_t b = ((int64_t)blockIdx.x * kWpb + wib) * 2 + cx.grp;
  const bool ghost = b >= bt.B;
  if (ghost) b = bt.B - 1;
  if (((int64_t)blockIdx.x * kWpb + wib) * 2 >= bt.B) return;  // whole warp beyond the batch
  double *wbase = smem + (size_t)wib * GSmem<N>::warp_total;
  double *base = wbase + MAT + (size_t)cx.grp * GSmem<N>::total;
  cx.SG = wbase;  // both series of the warp share the model
  cx.S0 = base; cx.S1 = base + MAT; cx.S2 = base + 2 * MAT; cx.S3 = base + 3 * MAT;
  double *v = base + GSmem<N>::kMats * MAT;
  cx.VA = v; cx.VB = v + VEC; cx.VX = v + 2 * VEC; cx.VK = v + 3 * VEC;
  cx.VD = v + 4 * VEC; cx.VZ = v + 5 * VEC;
  (void)sib;
  const int j = cx.jj;
  const bool wr = cx.act && !ghost;  // lane may write global memory
  const int T = bt.T, rows = T + 1;
  int st = 0;
  double Fk[N];  // F (n x 1), shared model

  // ---- per-series parameters
  const double V = bt.V.ptr[b * bt.V.sb];
  const double *wcolp = bt.W.ptr + b * bt.W.sb + (int64_t)j * N * bt.W.sk;  // column j of W
  auto load_model = [&](int t, bool first) {
    if (bt.g_tv || first) {
      const double *g = bt.G + (bt.g_tv ? (int64_t)t * NN : 0);
      __syncwarp();  // the other series may still be reading the previous G
      if (cx.grp == 0) {
#pragma unroll
        for (int i = 0; i < N; ++i) cx.SG[i + j * LD] = g[i + j * N];
      }
    }
    if (bt.f_tv || first) {
      const double *f = bt.F + (bt.f_tv ? (int64_t)t * N : 0);
#pragma unroll
      for (int i = 0; i < N; ++i) Fk[i] = f[i];
    }
    __syncwarp();
  };
  load_model(0, true);

  double m_j = bt.m0.ptr[b * bt.m0.sb + j * bt.m0.sk];
  double Ccol[N];
  {
    const double *cp = bt.C0.ptr + b * bt.C0.sb;
#pragma unroll
    for (int i = 0; i < N; ++i) Ccol[i] = cp[(i + j * N) * bt.C0.sk];
  }
  double *spill = (OP == kOpFfbs) ? wa.spill + (size_t)b * rows * wa.spill_k : nullptr;
  const double nanv = __longlong_as_double(0x7ff8000000000000LL);

  auto store_vec = [&](const View &vw, int64_t row, double x) {
    if (vw.ptr && wr) st_stream(vw.ptr + b * vw.sb + row * vw.sr + j * vw.sk, x);
  };
  auto store_col = [&](const View &vw, int64_t row, const double (&col)[N]) {
    if (vw.ptr && wr) {
      double *p = vw.ptr + b * vw.sb + row * vw.sr;
#pragma unroll
      for (int i = 0; i < N; ++i) st_stream(p + (i + j * N) * vw.sk, col[i]);
    }
  };
  auto spill_row = [&](int64_t row, double mj, const double (&C)[N], double aj, const double (&R)[N]) {
    if (!spill || !wr) return;
    double *sp = spill + (size_t)row * wa.spill_k;
    sp[j] = mj; sp[N + NN + j] = aj;
#pragma unroll
    for (int i = 0; i < N; ++i) { sp[N + i + j * N] = C[i]; sp[2 * N + NN + i + j * N] = R[i]; }
  };

  // initialiseState (KalmanFilter.scala:112-118): row 0
  store_vec(wa.kf.m, 0, m_j); store_vec(wa.kf.a, 0, m_j);
  store_col(wa.kf.C, 0, Ccol); store_col(wa.kf.R, 0, Ccol);
  if (cx.gl == 0 && !ghost) {
    if (wa.kf.f.ptr) wa.kf.f.ptr[b * wa.kf.f.sb] = nanv;
    if (wa.kf.Q.ptr) wa.kf.Q.ptr[b * wa.kf.Q.sb] = nanv;
  }
  spill_row(0, m_j, Ccol, m_j, Ccol);

  // ------------------------------------------------------------------ forward filter
  for (int t = 0; t < T; ++t) {
    const int64_t row = t + 1;
    load_model(t, false);
    const double y = bt.y.ptr[b * bt.y.sb + (int64_t)t * bt.y.sr];
    const double dt = bt.dt ? bt.dt[t] : 1.0;
    double a_j, Rcol[N];
    if (dt == 0.0) {  // uniform: the time grid is shared by the batch
      a_j = m_j;
#pragma unroll
      for (int i = 0; i < N; ++i) Rcol[i] = Ccol[i];
    } else {
      // a = G m
      if (cx.act) cx.VA[j] = m_j;
      __syncwarp();
      {
        double acc = 0.0;
#pragma unroll
        for (int k = 0; k < N; ++k) {
          const double prod = cx.SG[j + k * LD] * cx.VA[k];
          acc = (k == 0) ? prod : acc + prod;
        }
        a_j = acc;
      }
      // R = (G C) G^T + W dt
      double t1[N];
      mm_sx<N, LD>(cx.SG, Ccol, t1);                      // column j of G C (C column in registers)
      __syncwarp();
      if (cx.act) {
#pragma unroll
        for (int i = 0; i < N; ++i) cx.S0[i + j * LD] = t1[i];
      }
      __syncwarp();
      mm_sy<N, LD>(cx.S0, cx.SG + j, LD, Rcol);           // (G C) x row j of G
#pragma unroll
      for (int i = 0; i < N; ++i) Rcol[i] = Rcol[i] + wcolp[i * bt.W.sk] * dt;
    }
    // f = F^T a ; Q = (F^T R) F + V
    __syncwarp();
    if (cx.act) cx.VB[j] = a_j;
    double fr = 0.0;
#pragma unroll
    for (int k = 0; k < N; ++k) {
      const double prod = Fk[k] * Rcol[k];
      fr = (k == 0) ? prod : fr + prod;
    }
    if (cx.act) {
      cx.VX[j] = fr;
#pragma unroll
      for (int i = 0; i < N; ++i) cx.S1[i + j * LD] = Rcol[i];
    }
    __syncwarp();
    double f = 0.0, Q = 0.0;
#pragma unroll
    for (int k = 0; k < N; ++k) {
      const double pf = Fk[k] * cx.VB[k];
      f = (k == 0) ? pf : f + pf;
      const double pq = cx.VX[k] * Fk[k];
      Q = (k == 0) ? pq : Q + pq;
    }
    Q = Q + V;
    const bool obs = !isnan(y);
    // update (Joseph form), computed unconditionally and selected by `obs`
    double rhs_j = 0.0;
#pragma unroll
    for (int k = 0; k < N; ++k) {
      const double prod = Fk[k] * cx.S1[j + k * LD];
      rhs_j = (k == 0) ? prod : rhs_j + prod;
    }
    if (obs && Q == 0.0) st |= BDLM_ST_SINGULAR;
    const double K_j = rhs_j / Q;
    const double e = y - f;
    const double mn_j = a_j + K_j * e;
    if (cx.act) cx.VK[j] = K_j;
    __syncwarp();
    double Dcol[N], t1[N], Cn[N];
    double F_j = Fk[0];  // F element of this lane's column index
#pragma unroll
    for (int i = 1; i < N; ++i) F_j = (j == i) ? Fk[i] : F_j;
#pragma unroll
    for (int i = 0; i < N; ++i) Dcol[i] = ((i == j) ? 1.0 : 0.0) - cx.VK[i] * F_j;
    if (cx.act) {
#pragma unroll
      for (int i = 0; i < N; ++i) cx.S0[i + j * LD] = Dcol[i];
    }
    __syncwarp();
    mm_sy<N, LD>(cx.S0, cx.S1 + j * LD, 1, t1);  // D R   (S1 holds R)
    __syncwarp();
    if (cx.act) {
#pragma unroll
      for (int i = 0; i < N; ++i) cx.S2[i + j * LD] = t1[i];
    }
    __syncwarp();
    mm_sy<N, LD>(cx.S2, cx.S0 + j, LD, Cn);  // (D R) D^T : row j of D from S0
#pragma unroll
    for (int i = 0; i < N; ++i) Cn[i] = Cn[i] + (cx.VK[i] * V) * K_j;
    m_j = obs ? mn_j : a_j;
#pragma unroll
    for (int i = 0; i < N; ++i) Ccol[i] = obs ? Cn[i] : Rcol[i];
    store_vec(wa.kf.a, row, a_j); store_col(wa.kf.R, row, Rcol);
    store_vec(wa.kf.m, row, m_j); store_col(wa.kf.C, row, Ccol);
    if (cx.gl == 0 && !ghost) {
      if (wa.kf.f.ptr) st_stream(wa.kf.f.ptr + b * wa.kf.f.sb + row * wa.kf.f.sr, f);
      if (wa.kf.Q.ptr) st_stream(wa.kf.Q.ptr + b * wa.kf.Q.sb + row * wa.kf.Q.sr, Q);
    }
    spill_row(row, m_j, Ccol, a_j, Rcol);
    __syncwarp();
  }

  // ------------------------------------------------------------------ backward sampling
  double th_j = 0.0;
  if (OP == kOpFfbs) {
    // initialise (Smoothing.scala:105-109): theta_T ~ N(m_T, C_T)
    __syncwarp();
    if (cx.act) {
#pragma unroll
      for (int i = 0; i < N; ++i) cx.S0[i + j * LD] = Ccol[i];
    }
    __syncwarp();
    {
      const double z = wa.z.ptr ? wa.z.ptr[b * wa.z.sb + (int64_t)(rows - 1) * wa.z.sr + j * wa.z.sk]
                                : philox_normal(RngKey{wa.rng_seed, wa.rng_sweep}, wa.rng_base + b, rows, rows - 1, N, j);
      th_j = eig_draw<N>(cx, m_j, z, st);
    }
    store_vec(wa.theta, rows - 1, th_j);
    if (spill) __threadfence_block();
    for (int r = rows - 2; r >= 0; --r) {
      const int tobs = r;  // observation index of row r + 1 (keep_init = 1)
      load_model(tobs, false);
      const double dt = bt.dt ? bt.dt[tobs] : 1.0;
      const double *sp = spill + (size_t)r * wa.spill_k, *sp1 = sp + wa.spill_k;
      __syncwarp();
      // C_t -> S0, R_{t+1} -> S1 (both needed by rows and by columns)
      double Ccur[N], Arow[N];
#pragma unroll
      for (int i = 0; i < N; ++i) {
        Ccur[i] = sp[N + i + j * N];
        const double rv = sp1[2 * N + NN + i + j * N];
        if (cx.act) { cx.S0[i + j * LD] = Ccur[i]; cx.S1[i + j * LD] = rv; }
      }
      m_j = sp[j];
      const double a1_j = sp1[N + NN + j];
      const double z = wa.z.ptr ? wa.z.ptr[b * wa.z.sb + (int64_t)r * wa.z.sr + j * wa.z.sk]
                                : philox_normal(RngKey{wa.rng_seed, wa.rng_sweep}, wa.rng_base + b, rows, r, N, j);
      __syncwarp();
#pragma unroll
      for (int k = 0; k < N; ++k) Arow[k] = cx.S1[j + k * LD];
      // B = (R1^T \ (G C^T))^T
      double X[N];
      mm_sy<N, LD>(cx.SG, cx.S0 + j, LD, X);  // column j of G C^T (row j of C from S0)
      st |= lu_cols<N>(cx, Arow, X);  // X = column j of the solution = row j of B
      // B -> S3
      if (cx.act) {
#pragma unroll
        for (int c = 0; c < N; ++c) cx.S3[j + c * LD] = X[c];
        cx.VD[j] = th_j - a1_j;
      }
      __syncwarp();
      double h_j;
      {
        double acc = 0.0;
#pragma unroll
        for (int k = 0; k < N; ++k) {
          const double prod = X[k] * cx.VD[k];
          acc = (k == 0) ? prod : acc + prod;
        }
        h_j = m_j + acc;
      }
      // diff = I - B G
      double t1[N], Dcol[N], H1[N], H2[N];
      mm_sy<N, LD>(cx.S3, cx.SG + j * LD, 1, t1);   // B x column j of G
#pragma unroll
      for (int i = 0; i < N; ++i) Dcol[i] = ((i == j) ? 1.0 : 0.0) - t1[i];
      if (cx.act) {
#pragma unroll
        for (int i = 0; i < N; ++i) cx.S2[i + j * LD] = Dcol[i];
      }
      __syncwarp();
      mm_sy<N, LD>(cx.S2, cx.S0 + j * LD, 1, t1);  // diff C   (column j of C_t from S0)
      __syncwarp();
      if (cx.act) {
#pragma unroll
        for (int i = 0; i < N; ++i) cx.S0[i + j * LD] = t1[i];
      }
      __syncwarp();
      mm_sy<N, LD>(cx.S0, cx.S2 + j, LD, H1);      // (diff C) diff^T : row j of diff from S2
      mm_sy<N, LD>(cx.S3, wcolp, bt.W.sk, t1);     // B W : column j of W
#pragma unroll
      for (int i = 0; i < N; ++i) t1[i] = t1[i] * dt;
      __syncwarp();
      if (cx.act) {
#pragma unroll
        for (int i = 0; i < N; ++i) cx.S1[i + j * LD] = t1[i];
      }
      __syncwarp();
      mm_sy<N, LD>(cx.S1, cx.S3 + j, LD, H2);  // ((B W) dt) B^T : column j of B^T = row j of B
      __syncwarp();
      if (cx.act) {
#pragma unroll
        for (int i = 0; i < N; ++i) cx.S2[i + j * LD] = H1[i] + H2[i];
      }
      __syncwarp();
      double Hs[N];
#pragma unroll
      for (int i = 0; i < N; ++i) Hs[i] = (cx.S2[i + j * LD] + cx.S2[j + i * LD]) / 2.0;
      __syncwarp();
      if (cx.act) {
#pragma unroll
        for (int i = 0; i < N; ++i) cx.S0[i + j * LD] = Hs[i];
      }
      __syncwarp();
      th_j = eig_draw<N>(cx, h_j, z, st);
      store_vec(wa.theta, r, th_j);
    }
  }

  // ------------------------------------------------------------------ Gibbs statistics
  if (OP == kOpFfbs &&
      (wa.stats.ssy.ptr || wa.stats.ny.ptr || wa.stats.ssw.ptr || wa.stats.scatter.ptr)) {
    __syncwarp();
    double ssy = 0.0, ny = 0.0, ssw = 0.0, sc[N];
    const View &th = wa.theta;
    double prev_j = th.ptr[b * th.sb + j * th.sk];  // theta_0 (written by this lane)
    for (int t = 0; t < T; ++t) {
      load_model(t, false);
      const double cur_j = th.ptr[b * th.sb + (int64_t)(t + 1) * th.sr + j * th.sk];
      const double y = bt.y.ptr[b * bt.y.sb + (int64_t)t * bt.y.sr];
      const double dt = bt.dt ? bt.dt[t] : 1.0;
      if (cx.act) { cx.VA[j] = cur_j; cx.VB[j] = prev_j; }
      __syncwarp();
      double ft = 0.0, gx = 0.0;
#pragma unroll
      for (int k = 0; k < N; ++k) {
        const double pf = Fk[k] * cx.VA[k];
        ft = (k == 0) ? pf : ft + pf;
        const double pg = cx.SG[j + k * LD] * cx.VB[k];
        gx = (k == 0) ? pg : gx + pg;
      }
      double res = 0.0;
      if (!isnan(y)) { const double d = y - ft; res = d * d; ny += 1.0; }
      ssy = (t == 0) ? res : ssy + res;
      const double d_j = cur_j - gx;
      if (cx.act) cx.VD[j] = d_j;
      const double vw = (d_j * d_j) / dt;
      ssw = (t == 0) ? vw : ssw + vw;
      __syncwarp();
#pragma unroll
      for (int i = 0; i < N; ++i) {
        const double vv = (cx.VD[i] * d_j) / dt;
        sc[i] = (t == 0) ? vv : sc[i] + vv;
      }
      prev_j = cur_j;
      __syncwarp();
    }
    const StatViews &sv = wa.stats;
    if (cx.gl == 0 && !ghost) {
      if (sv.ssy.ptr) sv.ssy.ptr[b * sv.ssy.sb] = ssy;
      if (sv.ny.ptr) sv.ny.ptr[b * sv.ny.sb] = ny;
    }
    if (wr) {
      if (sv.ssw.ptr) sv.ssw.ptr[b * sv.ssw.sb + j * sv.ssw.sk] = ssw;
      if (sv.scatter.ptr) {
#pragma unroll
        for (int i = 0; i < N; ++i) sv.scatter.ptr[b * sv.scatter.sb + (i + j * N) * sv.scatter.sk] = sc[i];
      }
    }
  }

  if (bt.status) {
    const double chk = (OP == kOpFfbs) ? th_j : m_j;
    const bool bad = cx.act && !isfinite(chk);
    const unsigned bal = __ballot_sync(FULL, bad);
    // status bits raised by any lane of the group
    int stg = st;
#pragma unroll
    for (int off = GW / 2; off >= 1; off >>= 1) stg |= __shfl_xor_sync(FULL, stg, off);
    if (((bal >> (cx.grp * GW)) & 0xffffu) != 0) stg |= BDLM_ST_NONFINITE;
    if (cx.gl == 0 && !ghost) bt.status[b] = stg;
  }
}

template <int N, int OP>
cudaError_t launch_group_n(const WarpArgs &wa, cudaStream_t stream) {
  const size_t smem = (size_t)kWpb * GSmem<N>::warp_total * sizeof(double);
  cudaError_t e = cudaFuncSetAttribute(group_kernel<N, OP>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const int64_t per_block = kWpb * 2;
  const int64_t blocks = (wa.bt.B + per_block - 1) / per_block;
  if (blocks <= 0) return cudaSuccess;
  group_kernel<N, OP><<<(unsigned)blocks, kWpb * 32, smem, stream>>>(wa);
  return cudaGetLastError();
}

}  // namespace

// Shapes served by the two-series-per-warp kernels: p = 1, keep_init = 1, n in {7, 13}
// (polynomial(1) |+| seasonal(24, 3) and (24, 6): SeasonalModel.scala:14 and config 3).
bool group_supported(int op, int n, int p, int keep_init) {
  return (op == kOpFfbs || op == kOpFilter) && p == 1 && keep_init == 1 && (n == 13 || n == 7);
}

cudaError_t launch_group(int op, const WarpArgs &wa, cudaStream_t stream) {
  const int n = wa.bt.n;
  if (op == kOpFfbs) {
    if (n == 13) return launch_group_n<13, kOpFfbs>(wa, stream);
    if (n == 7) return launch_group_n<7, kOpFfbs>(wa, stream);
  } else if (op == kOpFilter) {
    if (n == 13) return launch_group_n<13, kOpFilter>(wa, stream);
    if (n == 7) return launch_group_n<7, kOpFilter>(wa, stream);
  }
  return cudaErrorInvalidValue;
}

}  // namespace bdlm
