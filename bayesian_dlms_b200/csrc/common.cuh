// common.cuh -- shared device/host definitions for libbdlm.so (sm_100a only).
//
// Arithmetic contract (DESIGN.md "Parity"): every kernel performs the reference's fp64
// operations in the reference's order with NO fused multiply-add (the JVM never fuses),
// so results are bit-identical to oracle/bdlm_oracle.c.  This translation unit set is
// therefore compiled with -fmad=false; do not introduce fma()/__fma_rn() calls.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/bdlm.h"

namespace bdlm {

// Strided view of a per-step array: element (series b, row r, component k) lives at
// ptr[b * sb + r * sr + k * sk].  ptr == nullptr means "not wanted".
struct View {
  double *ptr;
  int64_t sb, sr, sk;
};
struct CView {
  const double *ptr;
  int64_t sb, sr, sk;
};

// Per-series parameter view: element (b, k) at ptr[b * sb + k * sk]; sb = 0 when the
// parameter is shared by the batch.
struct PView {
  const double *ptr;
  int64_t sb, sk;
};

struct KfViews {
  View m, C, a, R, f, Q;
};

// Launch description shared by all kernels.
struct Batch {
  int64_t B;       // series in this launch
  int T;           // observations
  int n, p;
  int keep_init;   // rows = T + keep_init
  int compat;      // BDLM_TEXTBOOK_* | BDLM_SVD_*
  const double *F; // device [n*p] or [T][n*p]; per series: element (b, t, k) at F[b*F_sb + t*F_sr + k*F_sk]
  const double *G; // device [n*n] or [T][n*n]; per series: G[b*G_sb + t*G_sr + k*G_sk]
  const double *dt;// device (dt into observation t) or nullptr = all 1.0; element (b, t) at
                   // dt[b*dt_sb + t*dt_sr] -- shared by the batch: dt_sb = 0, dt_sr = 1
  int64_t dt_sb, dt_sr;
  int64_t F_sb, F_sr, F_sk, G_sb, G_sr, G_sk;  // shared: sb = 0, sr = (tv ? k : 0), sk = 1
  int ps_model;    // F or G given per series (Data.time / regression covariates differ by series)
  int f_tv, g_tv;
  int v_tv;        // V varies with t (StudentTGibbs.filter): V holds T matrices, row stride V_sr
  int64_t V_sr;
  int w_tv;        // W varies with t (DlmFsvSystem.ffbs): W holds T matrices, row stride W_sr
  int64_t W_sr;
  PView V, W, m0, C0;
  CView y;         // T rows
  int32_t *status; // [B] or nullptr
};

// dt into observation t of series b (1.0 on the regular grid)
__device__ __forceinline__ double dt_at(const Batch &bt, int64_t b, int t) {
  return bt.dt ? bt.dt[b * bt.dt_sb + (int64_t)t * bt.dt_sr] : 1.0;
}

__host__ __device__ inline int64_t vidx(int64_t sb, int64_t sr, int64_t sk, int64_t b,
                                        int64_t r, int64_t k) {
  return b * sb + r * sr + k * sk;
}

// Streaming (evict-first) store: outputs are written once and never re-read by the
// same kernel except the (m, C) spill, which is stored with default policy.  Other cache
// policies measured no different (profiles/r1_tuning.txt, "store / load cache policy").
__device__ __forceinline__ void st_stream(double *p, double v) { __stcs(p, v); }
__device__ __forceinline__ double ld_stream(const double *p) { return __ldcs(p); }

constexpr double kJacobiThr2 = 1e-30; // rotate iff a_pq^2 > (1e-15)^2 |a_pp a_qq|
constexpr int kJacobiMaxSweeps = 30;

}  // namespace bdlm
