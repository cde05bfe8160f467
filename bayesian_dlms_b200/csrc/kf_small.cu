// kf_small.cu -- register-resident Kalman filter + RTS smoother for small state
// dimension (n <= 4, p = 1): ONE THREAD PER SERIES.
//
// This is the HBM-bound headline kernel (BASELINE.json config 2: polynomial(2), 1e6
// series x T = 1000).  Per series-step it moves 8*(p + 2n + 2n^2 + p + p^2) bytes in the
// forward pass and 8*(2n + 2n^2) in the backward pass (216 B for n = 2, p = 1) against
// ~130 flops, so everything is organised around HBM:
//   * device-native layout is time-major SoA [rows][k][B]: the 32 threads of a warp read
//     or write 256 contiguous bytes per scalar field per step (two full 128 B lines),
//   * the whole state (m, C, a, R, W, s, S) lives in registers, the shared model (F, G)
//     in the kernel-parameter constant bank,
//   * y is prefetched one 4-step chunk ahead and the backward pass's (m_t, C_t) one row
//     ahead, so every thread always has independent loads in flight while it walks its
//     strictly sequential recursion,
//   * outputs are written once with streaming stores (evict-first) and a_{t+1}, R_{t+1}
//     are recomputed in the backward pass (bit-identical to the forward values) instead
//     of being re-read.
//
// Arithmetic mirrors oracle/bdlm_oracle.c operation for operation (see common.cuh);
// reference citations: KalmanFilter.scala:64-107,273-321 and Smoothing.scala:31-64.
#include "common.cuh"
#include "launch.h"
#include "small_steps.cuh"

namespace bdlm {

namespace {

using namespace small;

template <int K>
__device__ __forceinline__ void store_vec(const View &v, int64_t b, int64_t row,
                                          const double *x) {
  if (v.ptr == nullptr) return;
  double *p = v.ptr + b * v.sb + row * v.sr;
#pragma unroll
  for (int k = 0; k < K; ++k) st_stream(p + k * v.sk, x[k]);
}

template <int K>
__device__ __forceinline__ void load_vec(const View &v, int64_t b, int64_t row, double *x) {
  const double *p = v.ptr + b * v.sb + row * v.sr;
#pragma unroll
  for (int k = 0; k < K; ++k) x[k] = ld_stream(p + k * v.sk);
}

// (prefetch.global.L2 of the spill rows 3 or 6 iterations ahead was measured 5 % SLOWER on
// B200 and removed -- profiles/r1_tuning.txt; the backward pass uses a cp.async ring instead.)

template <int K>
__device__ __forceinline__ void load_param(const PView &v, int64_t b, double *x) {
  const double *p = v.ptr + b * v.sb;
#pragma unroll
  for (int k = 0; k < K; ++k) x[k] = p[k * v.sk];
}

template <int N>
struct SmallModel {
  double G[N * N];
  double F[N];
};

// Model matrices for observation t: kernel-parameter constant bank when time-invariant
// (static indices, no address taken), uniform global loads when they vary with t.
template <int N, bool REG>
__device__ __forceinline__ void load_model(const Batch &bt, const SmallModel<N> &mdl, int64_t b, int t,
                                           double (&G)[N * N], double (&F)[N]) {
  if (!REG && bt.g_tv) {  // shared [T][n*n] (uniform loads) or per series (coalesced, time-major)
    const double *g = bt.G + b * bt.G_sb + (int64_t)t * bt.G_sr;
#pragma unroll
    for (int k = 0; k < N * N; ++k) G[k] = __ldg(g + k * bt.G_sk);
  } else {
#pragma unroll
    for (int k = 0; k < N * N; ++k) G[k] = mdl.G[k];
  }
  if (!REG && bt.f_tv) {
    const double *f = bt.F + b * bt.F_sb + (int64_t)t * bt.F_sr;
#pragma unroll
    for (int k = 0; k < N; ++k) F[k] = __ldg(f + k * bt.F_sk);
  } else {
#pragma unroll
    for (int k = 0; k < N; ++k) F[k] = mdl.F[k];
  }
}

constexpr int kChunk = 4;  // y prefetch distance (steps)
constexpr int kRing = 4;   // backward-pass spill rows in flight per thread (power of two)

__device__ __forceinline__ void cp_async8(double *smem_dst, const double *gmem_src) {
  const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(sa), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int K>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(K) : "memory"); }

// mode bits (compile-time: a runtime branch between "recompute a,R" and "reload a,R" made
// ptxas put the prefetch loads and the reload loads on one scoreboard slot and wait for it
// at the merge point, which serialised the (m, C) prefetch with the recursion)
constexpr int kDoFilter = 1, kDoSmooth = 2;

// Minimum resident blocks per SM asked of ptxas (register cap = 65536 / (128 * blocks)).
// n = 2: profiles/r1_tuning.txt, kf_small_kernel table ("minBlocks=5 ... chosen"); n = 3, 4:
// profiles/r2_tuning.txt, "register kernels away from n = 2".
template <int N> struct Occ { static constexpr int kMinBlocks = 1; };
template <> struct Occ<1> { static constexpr int kMinBlocks = 6; };
template <> struct Occ<2> { static constexpr int kMinBlocks = 5; };
template <> struct Occ<3> { static constexpr int kMinBlocks = 3; };
template <> struct Occ<4> { static constexpr int kMinBlocks = 1; };

template <int N, bool REG, int MODE, bool RELOAD>
__global__ void __launch_bounds__(128, Occ<N>::kMinBlocks)
kf_small_kernel(const Batch bt, const SmallModel<N> mdl, const KfViews kf, const View sv,
                const View Sv) {
  const int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (b >= bt.B) return;
  const int T = bt.T, ki = bt.keep_init, rows = T + ki;
  int st = 0;

  double W[N * N], m[N], C[N * N];
  double V;
  load_param<N * N>(bt.W, b, W);
  load_param<1>(bt.V, b, &V);

  if (MODE & kDoFilter) {
    load_param<N>(bt.m0, b, m);
    load_param<N * N>(bt.C0, b, C);
    if (ki) {  // initialiseState (KalmanFilter.scala:112-118): f, Q = None -> NaN
      const double nanv = __longlong_as_double(0x7ff8000000000000LL);
      store_vec<N>(kf.m, b, 0, m);
      store_vec<N * N>(kf.C, b, 0, C);
      store_vec<N>(kf.a, b, 0, m);
      store_vec<N * N>(kf.R, b, 0, C);
      store_vec<1>(kf.f, b, 0, &nanv);
      store_vec<1>(kf.Q, b, 0, &nanv);
    }
    const double *yp = bt.y.ptr + b * bt.y.sb;
    double ycur[kChunk], ynxt[kChunk];
#pragma unroll
    for (int u = 0; u < kChunk; ++u) ycur[u] = (u < T) ? ld_stream(yp + u * bt.y.sr) : 0.0;
    for (int t0 = 0; t0 < T; t0 += kChunk) {
#pragma unroll
      for (int u = 0; u < kChunk; ++u) {
        const int t = t0 + kChunk + u;
        ynxt[u] = (t < T) ? ld_stream(yp + (int64_t)t * bt.y.sr) : 0.0;
      }
#pragma unroll
      for (int u = 0; u < kChunk; ++u) {
        const int t = t0 + u;
        if (t < T) {
          double a[N], R[N * N], f, Q;
          const double dt = REG ? 1.0 : dt_at(bt, b, t);
          double G[N * N], F[N];
          load_model<N, REG>(bt, mdl, b, t, G, F);
          advance<N, REG>(G, W, dt, m, C, a, R);
          update<N>(F, V, ycur[u], a, R, f, Q, m, C, st);
          const int64_t row = t + ki;
          store_vec<N>(kf.a, b, row, a);
          store_vec<N * N>(kf.R, b, row, R);
          store_vec<1>(kf.f, b, row, &f);
          store_vec<1>(kf.Q, b, row, &Q);
          store_vec<N>(kf.m, b, row, m);
          store_vec<N * N>(kf.C, b, row, C);
        }
      }
#pragma unroll
      for (int u = 0; u < kChunk; ++u) ycur[u] = ynxt[u];
    }
  } else {
    load_vec<N>(kf.m, b, rows - 1, m);
    load_vec<N * N>(kf.C, b, rows - 1, C);
  }

  if (MODE & kDoSmooth) {
    // backwardsSmoother (Smoothing.scala:57-64): s_T = m_T, S_T = C_T
    double s[N], S[N * N];
#pragma unroll
    for (int i = 0; i < N; ++i) s[i] = m[i];
#pragma unroll
    for (int k = 0; k < N * N; ++k) S[k] = C[k];
    store_vec<N>(sv, b, rows - 1, s);
    store_vec<N * N>(Sv, b, rows - 1, S);
    const bool textbook = (bt.compat & BDLM_TEXTBOOK_SMOOTHER) != 0;
    // (m_t, C_t) spill rows are staged through a per-thread shared-memory ring by cp.async
    // (LDGSTS), kRing rows deep: the loads bypass the register file and the scoreboard, so
    // they stay in flight across several iterations of the recursion.  (One row of register
    // prefetch was not enough: ncu showed 25 % of all stall samples on its first use; DRAM
    // latency under this kernel's write-heavy load exceeds one backward iteration.)
    extern __shared__ double ring[];
    constexpr int kRow = N + N * N;
    const int nthr = blockDim.x;
    auto slot = [&](int r, int k) { return ring + ((size_t)(r & (kRing - 1)) * kRow + k) * nthr + threadIdx.x; };
    auto issue = [&](int r) {
      if (r >= 0) {
        const double *pm = kf.m.ptr + b * kf.m.sb + (int64_t)r * kf.m.sr;
        const double *pc = kf.C.ptr + b * kf.C.sb + (int64_t)r * kf.C.sr;
#pragma unroll
        for (int k = 0; k < N; ++k) cp_async8(slot(r, k), pm + k * kf.m.sk);
#pragma unroll
        for (int k = 0; k < N * N; ++k) cp_async8(slot(r, N + k), pc + k * kf.C.sk);
      }
      cp_async_commit();
    };
    double an[N], Rn[N * N];
#pragma unroll
    for (int d = 0; d < kRing - 1; ++d) issue(rows - 2 - d);
    if (RELOAD && rows >= 2) {
      load_vec<N>(kf.a, b, rows - 1, an);
      load_vec<N * N>(kf.R, b, rows - 1, Rn);
    }
    for (int r = rows - 2; r >= 0; --r) {
      double a1[N], R1[N * N];
      issue(r - (kRing - 1));
      cp_async_wait<kRing - 1>();  // the group of row r has landed
#pragma unroll
      for (int i = 0; i < N; ++i) m[i] = *slot(r, i);
#pragma unroll
      for (int k = 0; k < N * N; ++k) C[k] = *slot(r, N + k);
      if (RELOAD) {
#pragma unroll
        for (int i = 0; i < N; ++i) a1[i] = an[i];
#pragma unroll
        for (int k = 0; k < N * N; ++k) R1[k] = Rn[k];
        if (r > 0) {
          load_vec<N>(kf.a, b, r, an);
          load_vec<N * N>(kf.R, b, r, Rn);
        }
      }
      const int tobs = r + 1 - ki;  // observation index of row r + 1
      const double dt = REG ? 1.0 : dt_at(bt, b, tobs);
      double G[N * N], F[N];
      load_model<N, REG>(bt, mdl, b, tobs, G, F);
      if (!RELOAD) advance<N, REG>(G, W, dt, m, C, a1, R1);  // bit-identical to the forward a, R
      rts_step<N>(G, m, C, a1, R1, textbook, s, S, st);
      store_vec<N>(sv, b, r, s);
      store_vec<N * N>(Sv, b, r, S);
    }
#pragma unroll
    for (int i = 0; i < N; ++i) m[i] = s[i];
#pragma unroll
    for (int k = 0; k < N * N; ++k) C[k] = S[k];
  }

  if (bt.status) {
    bool finite = true;
#pragma unroll
    for (int i = 0; i < N; ++i) finite = finite && isfinite(m[i]);
#pragma unroll
    for (int k = 0; k < N * N; ++k) finite = finite && isfinite(C[k]);
    if (!finite) st |= BDLM_ST_NONFINITE;
    bt.status[b] = st;
  }
}

constexpr int kThreads = 128;

template <int N, bool REG, int MODE, bool RELOAD>
cudaError_t launch_t(const Batch &bt, const SmallModel<N> &mdl, const KfViews &kf, const View &sv,
                     const View &Sv, cudaStream_t stream, int *wave_series) {
  if (wave_series) {  // occupancy query only
    int blocks = 0, dev = 0, sms = 0;
    const size_t qsmem = (MODE & kDoSmooth) ? sizeof(double) * kRing * (N + N * N) * kThreads : 0;
    if (qsmem > 48 * 1024) {  // n = 4: 80 KB ring -- the query needs the opt-in limit raised first
      cudaError_t ea = cudaFuncSetAttribute(kf_small_kernel<N, REG, MODE, RELOAD>,
                                            cudaFuncAttributeMaxDynamicSharedMemorySize, (int)qsmem);
      if (ea != cudaSuccess) return ea;
    }
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(
        &blocks, kf_small_kernel<N, REG, MODE, RELOAD>, kThreads, qsmem);
    if (e != cudaSuccess) return e;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    *wave_series = blocks * sms * kThreads;
    return cudaSuccess;
  }
  const int64_t blocks = (bt.B + kThreads - 1) / kThreads;
  if (blocks <= 0) return cudaSuccess;
  const size_t smem = (MODE & kDoSmooth) ? sizeof(double) * kRing * (N + N * N) * kThreads : 0;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kf_small_kernel<N, REG, MODE, RELOAD>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  kf_small_kernel<N, REG, MODE, RELOAD><<<(unsigned)blocks, kThreads, smem, stream>>>(bt, mdl, kf, sv, Sv);
  return cudaGetLastError();
}

template <int N>
cudaError_t launch_n(const Batch &bt, const double *hG, const double *hF, const KfViews &kf,
                     const View &sv, const View &Sv, int mode, cudaStream_t stream,
                     int *wave_series) {
  SmallModel<N> mdl;
  for (int k = 0; k < N * N; ++k) mdl.G[k] = hG ? hG[k] : 0.0;
  for (int k = 0; k < N; ++k) mdl.F[k] = hF ? hF[k] : 0.0;
  const bool reg = bt.dt == nullptr && !bt.g_tv && !bt.f_tv;
  const bool reload = mode == kDoSmooth && kf.a.ptr != nullptr && kf.R.ptr != nullptr;
#define BDLM_GO(REG_, MODE_, RELOAD_) \
  return launch_t<N, REG_, MODE_, RELOAD_>(bt, mdl, kf, sv, Sv, stream, wave_series)
  if (mode == kDoFilter) { if (reg) BDLM_GO(true, kDoFilter, false); else BDLM_GO(false, kDoFilter, false); }
  if (mode == (kDoFilter | kDoSmooth)) {
    if (reg) BDLM_GO(true, kDoFilter | kDoSmooth, false); else BDLM_GO(false, kDoFilter | kDoSmooth, false);
  }
  if (reload) { if (reg) BDLM_GO(true, kDoSmooth, true); else BDLM_GO(false, kDoSmooth, true); }
  if (reg) BDLM_GO(true, kDoSmooth, false); else BDLM_GO(false, kDoSmooth, false);
#undef BDLM_GO
}

}  // namespace

bool small_supported(int n, int p) { return p == 1 && n >= 1 && n <= 4; }

cudaError_t launch_kf_small(const Batch &bt, const double *hG, const double *hF,
                            const KfViews &kf, const View &sv, const View &Sv,
                            bool do_filter, bool do_smooth, cudaStream_t stream,
                            int *wave_series) {
  const int mode = (do_filter ? kDoFilter : 0) | (do_smooth ? kDoSmooth : 0);
  switch (bt.n) {
    case 1: return launch_n<1>(bt, hG, hF, kf, sv, Sv, mode, stream, wave_series);
    case 2: return launch_n<2>(bt, hG, hF, kf, sv, Sv, mode, stream, wave_series);
    case 3: return launch_n<3>(bt, hG, hF, kf, sv, Sv, mode, stream, wave_series);
    case 4: return launch_n<4>(bt, hG, hF, kf, sv, Sv, mode, stream, wave_series);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace bdlm
