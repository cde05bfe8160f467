// kf_small.cu -- register-resident Kalman filter + RTS smoother for small state
// dimension (n <= 4, p = 1): ONE THREAD PER SERIES.
//
// This is the HBM-bound headline kernel (BASELINE.json config 2: polynomial(2), 1e6
// series x T = 1000).  Per series-step the forward pass moves 8*(p + 2n + 2n^2 + p + p^2)
// bytes and the backward pass writes 8*(n + n^2) (s, S) and reads back what it needs of the
// forward pass: 8*(n + n^2) of (m_t, C_t), or, fused with the filter for n <= 2 on a regular grid, one
// checkpoint row of (m, C) in kSeg plus y again (186 B in all for n = 2, p = 1, against 216 B
// with the full re-read) against ~130 flops, so everything is organised around HBM:
//   * device-native layout is time-major SoA [rows][k][B]: the 32 threads of a warp read
//     or write 256 contiguous bytes per scalar field per step (two full 128 B lines),
//   * the whole state (m, C, a, R, W, s, S) lives in registers, the shared model (F, G)
//     in the kernel-parameter constant bank,
//   * y is prefetched one 4-step chunk ahead and the backward pass's rows are staged by
//     cp.async ahead of use, so every thread always has independent loads in flight while it
//     walks its strictly sequential recursion,
//   * outputs are written once with streaming stores (evict-first); the backward pass
//     recomputes a_{t+1}, R_{t+1} and, fused for n <= 2, the filtered (m_t, C_t) between
//     checkpoints (bit-identical to the forward values) instead of re-reading them.
//
// Arithmetic mirrors oracle/bdlm_oracle.c operation for operation (see common.cuh);
// reference citations: KalmanFilter.scala:64-107,273-321 and Smoothing.scala:31-64.
#include "common.cuh"
#include "launch.h"
#include "small_steps.cuh"

namespace bdlm {

namespace {

using namespace small;

// The time loops keep one address per field for the current row (row_ptr once, then a step of
// v.sr per row) and store at p + k * sk: a 64-bit add of a uniform offset per element instead of
// recomputing ptr + b * sb + row * sr + k * sk in 64-bit multiplies for every store.
__device__ __forceinline__ double *row_ptr(const View &v, int64_t b, int64_t row) {
  return v.ptr + b * v.sb + row * v.sr;
}

// p = row_ptr(v, b, row); a field the caller did not ask for (v.ptr == nullptr, a kernel
// parameter) costs one uniform branch per store, unless DENSE: every field is known to be wanted
template <bool DENSE, int K>
__device__ __forceinline__ void store_at(const View &v, double *p, const double *x) {
  if (!DENSE && v.ptr == nullptr) return;
#pragma unroll
  for (int k = 0; k < K; ++k) st_stream(p + k * v.sk, x[k]);
}

template <int K>
__device__ __forceinline__ void store_vec(const View &v, int64_t b, int64_t row,
                                          const double *x) {
  store_at<false, K>(v, row_ptr(v, b, row), x);
}

template <int K>
__device__ __forceinline__ void load_vec(const View &v, int64_t b, int64_t row, double *x) {
  const double *p = row_ptr(v, b, row);
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
// with kDoFilter | kDoSmooth: the caller wants all eight outputs, so the time loops store
// without testing each field's pointer (the benchmark's and the dense device path's call)
constexpr int kAllOut = 4;

// Minimum resident blocks per SM asked of ptxas (register cap = 65536 / (128 * blocks)).
// n = 2: profiles/r1_tuning.txt, kf_small_kernel table ("minBlocks=5 ... chosen"); n = 3, 4:
// profiles/r2_tuning.txt, "register kernels away from n = 2".
template <int N> struct Occ { static constexpr int kMinBlocks = 1; };
template <> struct Occ<1> { static constexpr int kMinBlocks = 6; };
template <> struct Occ<2> { static constexpr int kMinBlocks = 5; };
template <> struct Occ<3> { static constexpr int kMinBlocks = 3; };
template <> struct Occ<4> { static constexpr int kMinBlocks = 1; };

// Fused filter + smoother, n <= 2, regular grid and time-invariant model: the backward pass
// rebuilds (m_t, C_t) on chip from every kSeg-th stored row instead of re-reading every row
// (DESIGN.md §3).  The smooth-only modes have no y to re-filter with; n = 3, 4 are FP64-bound
// (profiles/r2_tuning.txt, "which roof?"); off the REG path the re-filtering loads dt, F, G a
// second time and per-series G measured 3.6 % slower with it (profiles/r3_recompute.txt): all of
// those keep re-reading through the kRing ring.  kSeg: profiles/r3_recompute.txt.
constexpr int kSeg = 4;
template <int N, bool REG, int MODE>
constexpr bool recompute() {
  return (MODE & (kDoFilter | kDoSmooth)) == (kDoFilter | kDoSmooth) && N <= 2 && REG;
}

// Shared memory per thread, in doubles: the re-read ring, or kSeg recomputed rows plus a staging
// slot for the next segment's checkpoint row and its kSeg - 1 y values.
template <int N, bool REG, int MODE>
constexpr int smem_doubles() {
  return !(MODE & kDoSmooth) ? 0
         : recompute<N, REG, MODE>() ? (kSeg + 1) * (N + N * N) + kSeg - 1
                                 : kRing * (N + N * N);
}

// Threads per block.  The shared-memory slots are indexed with it as a compile-time stride, so
// every slot of a thread is its base address plus an immediate offset.
constexpr int kThreads = 128;

template <int N, bool REG, int MODE, bool RELOAD>
__global__ void __launch_bounds__(kThreads, Occ<N>::kMinBlocks)
kf_small_kernel(const Batch bt, const SmallModel<N> mdl, const KfViews kf, const View sv,
                const View Sv) {
  constexpr bool kDense = (MODE & kAllOut) != 0;
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
    double *pm = row_ptr(kf.m, b, ki), *pC = row_ptr(kf.C, b, ki), *pa = row_ptr(kf.a, b, ki),
           *pR = row_ptr(kf.R, b, ki), *pf = row_ptr(kf.f, b, ki), *pQ = row_ptr(kf.Q, b, ki);
    double ycur[kChunk], ynxt[kChunk];
#pragma unroll
    for (int u = 0; u < kChunk; ++u) ycur[u] = (u < T) ? ld_stream(yp + u * bt.y.sr) : 0.0;
    for (int t0 = 0; t0 < T; t0 += kChunk) {
      yp += kChunk * bt.y.sr;
#pragma unroll
      for (int u = 0; u < kChunk; ++u) ynxt[u] = (t0 + kChunk + u < T) ? ld_stream(yp + u * bt.y.sr) : 0.0;
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
          store_at<kDense, N>(kf.a, pa, a);
          store_at<kDense, N * N>(kf.R, pR, R);
          store_at<kDense, 1>(kf.f, pf, &f);
          store_at<kDense, 1>(kf.Q, pQ, &Q);
          store_at<kDense, N>(kf.m, pm, m);
          store_at<kDense, N * N>(kf.C, pC, C);
          pa += kf.a.sr; pR += kf.R.sr; pf += kf.f.sr; pQ += kf.Q.sr; pm += kf.m.sr; pC += kf.C.sr;
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
    double *ps = row_ptr(sv, b, rows - 1), *pS = row_ptr(Sv, b, rows - 1);
    store_at<kDense, N>(sv, ps, s);
    store_at<kDense, N * N>(Sv, pS, S);
    const bool textbook = (bt.compat & BDLM_TEXTBOOK_SMOOTHER) != 0;
    extern __shared__ double ring[];
    constexpr int kRow = N + N * N;
    // Smoothing.smoothStep for row r from its filtered (mr, Cr): a_{r+1}, R_{r+1} are recomputed
    // (bit-identical to the forward values) unless the caller passed them (a1, R1 preset).
    auto smooth_row = [&](int r, const double (&mr)[N], const double (&Cr)[N * N], double (&a1)[N],
                          double (&R1)[N * N]) {
      const int tobs = r + 1 - ki;  // observation index of row r + 1
      const double dt = REG ? 1.0 : dt_at(bt, b, tobs);
      double G[N * N], F[N];
      load_model<N, REG>(bt, mdl, b, tobs, G, F);
      if (!RELOAD) advance<N, REG>(G, W, dt, mr, Cr, a1, R1);
      rts_step<N>(G, mr, Cr, a1, R1, textbook, s, S, st);
      ps -= sv.sr; pS -= Sv.sr;
      store_at<kDense, N>(sv, ps, s);
      store_at<kDense, N * N>(Sv, pS, S);
    };
    if constexpr (recompute<N, REG, MODE>()) {
      // Rows 0 .. rows - 2 in segments [r0, r0 + len), r0 a multiple of kSeg, top segment first
      // (the only one that may be short).  The stored row r0 is the segment's checkpoint; rows
      // r0 + 1 .. r0 + len - 1 are filtered again from it with the forward pass's operations on
      // the same inputs, so they come out bit for bit as stored, and nothing is stored.  They are
      // kept in shared memory as [j][k][thread] (no bank conflicts) and smoothed in descending
      // order.  The next segment's checkpoint and y values are staged by cp.async a segment
      // ahead, into slot kSeg: kRow doubles of (m, C), then kSeg - 1 y values.
      auto seg = [&](int j, int k) { return ring + ((size_t)j * kRow + k) * kThreads + threadIdx.x; };
      auto issue = [&](int r0, int len) {
        if (r0 >= 0) {
          const double *pcm = row_ptr(kf.m, b, r0), *pcC = row_ptr(kf.C, b, r0);
#pragma unroll
          for (int k = 0; k < N; ++k) cp_async8(seg(kSeg, k), pcm + k * kf.m.sk);
#pragma unroll
          for (int k = 0; k < N * N; ++k) cp_async8(seg(kSeg, N + k), pcC + k * kf.C.sk);
          const double *py = bt.y.ptr + b * bt.y.sb + (int64_t)(r0 + 1 - ki) * bt.y.sr;
#pragma unroll
          for (int j = 0; j < kSeg - 1; ++j)
            if (j < len - 1) cp_async8(seg(kSeg, kRow + j), py + j * bt.y.sr);
        }
        cp_async_commit();
      };
      if (rows >= 2) {
        int r0 = (rows - 2) / kSeg * kSeg;
        issue(r0, rows - 1 - r0);
        for (; r0 >= 0; r0 -= kSeg) {
          const int len = min(kSeg, rows - 1 - r0);
          double yv[kSeg - 1];
          cp_async_wait<0>();
#pragma unroll
          for (int i = 0; i < N; ++i) m[i] = *seg(kSeg, i);
#pragma unroll
          for (int k = 0; k < N * N; ++k) C[k] = *seg(kSeg, N + k);
#pragma unroll
          for (int j = 0; j < kSeg - 1; ++j) yv[j] = (j < len - 1) ? *seg(kSeg, kRow + j) : 0.0;
          issue(r0 - kSeg, kSeg);  // the staging slot is free again
#pragma unroll
          for (int j = 0; j < kSeg; ++j) {
            if (j >= len) break;
            if (j > 0) {  // filter row r0 + j (observation r0 + j - ki) from row r0 + j - 1
              const int t = r0 + j - ki;
              double a[N], R[N * N], f, Q;
              const double dt = REG ? 1.0 : dt_at(bt, b, t);
              double G[N * N], F[N];
              load_model<N, REG>(bt, mdl, b, t, G, F);
              advance<N, REG>(G, W, dt, m, C, a, R);
              update<N>(F, V, yv[j - 1], a, R, f, Q, m, C, st);
            }
#pragma unroll
            for (int i = 0; i < N; ++i) *seg(j, i) = m[i];
#pragma unroll
            for (int k = 0; k < N * N; ++k) *seg(j, N + k) = C[k];
          }
#pragma unroll
          for (int j = kSeg - 1; j >= 0; --j) {
            if (j < len) {
              double a1[N], R1[N * N];
#pragma unroll
              for (int i = 0; i < N; ++i) m[i] = *seg(j, i);
#pragma unroll
              for (int k = 0; k < N * N; ++k) C[k] = *seg(j, N + k);
              smooth_row(r0 + j, m, C, a1, R1);
            }
          }
        }
      }
    } else {
      // (m_t, C_t) rows are staged through a per-thread shared-memory ring by cp.async
      // (LDGSTS), kRing rows deep: the loads bypass the register file and the scoreboard, so
      // they stay in flight across several iterations of the recursion.  (One row of register
      // prefetch was not enough: ncu showed 25 % of all stall samples on its first use; DRAM
      // latency under this kernel's write-heavy load exceeds one backward iteration.)
      auto slot = [&](int r, int k) { return ring + ((size_t)(r & (kRing - 1)) * kRow + k) * kThreads + threadIdx.x; };
      auto issue = [&](int r) {
        if (r >= 0) {
          const double *pcm = row_ptr(kf.m, b, r), *pcC = row_ptr(kf.C, b, r);
#pragma unroll
          for (int k = 0; k < N; ++k) cp_async8(slot(r, k), pcm + k * kf.m.sk);
#pragma unroll
          for (int k = 0; k < N * N; ++k) cp_async8(slot(r, N + k), pcC + k * kf.C.sk);
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
        smooth_row(r, m, C, a1, R1);
      }
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

template <int N, bool REG, int MODE, bool RELOAD>
cudaError_t launch_t(const Batch &bt, const SmallModel<N> &mdl, const KfViews &kf, const View &sv,
                     const View &Sv, cudaStream_t stream, int *wave_series) {
  if (wave_series) {  // occupancy query only
    int blocks = 0, dev = 0, sms = 0;
    const size_t qsmem = sizeof(double) * smem_doubles<N, REG, MODE>() * kThreads;
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
  const size_t smem = sizeof(double) * smem_doubles<N, REG, MODE>() * kThreads;
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
  if (mode == (kDoFilter | kDoSmooth)) {  // m, C are always given (the library's workspace if not wanted)
    const bool all = kf.a.ptr && kf.R.ptr && kf.f.ptr && kf.Q.ptr && sv.ptr && Sv.ptr;
    constexpr int kFS = kDoFilter | kDoSmooth;
    if (all) { if (reg) BDLM_GO(true, kFS | kAllOut, false); else BDLM_GO(false, kFS | kAllOut, false); }
    if (reg) BDLM_GO(true, kFS, false); else BDLM_GO(false, kFS, false);
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
