// api.cu -- C ABI of libbdlm.so (include/bdlm.h): context, validation, model upload,
// kernel selection, layout handling and the host-buffer slab pipeline.
//
// Kernel selection: n <= 4, p = 1 filter / smoother calls go to the register kernels of
// kf_small.cu (device-native time-major SoA; series-major data is transposed on the
// device through context workspace); everything else goes to the warp-per-series
// kernels of kf_warp.cu, which address user arrays through strided views.
//
// There is no CPU path in this file: every entry point either launches CUDA kernels or
// fails with an error code.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include <nvtx3/nvToolsExt.h>  // header-only NVTX 3: no link dependency, no cost without a tool attached

#include "common.cuh"
#include "ctx_internal.h"
#include "launch.h"

using namespace bdlm;

struct bdlm_ctx {
  int device = 0;
  cudaStream_t own_stream = nullptr, stream = nullptr;
  cudaStream_t s_in = nullptr, s_out = nullptr;
  cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_comp[2] = {nullptr, nullptr},
              ev_out[2] = {nullptr, nullptr};
  std::string err;
  int64_t launches = 0;
  char *arena = nullptr;
  size_t arena_bytes = 0;
  size_t staging_cap = (size_t)8 << 30;
  size_t workspace_cap = (size_t)48 << 30;  // device-mode spill/transposes per launch
  unsigned long long rng_seed = 0, rng_sweep = 0;  // on-device RNG mode of the FFBS calls (z == NULL)
  long long rng_first = 0;                         // global index of a call's first series
  void *scan_table = nullptr;          // scan.cu forward table of the model in scan_key
  std::vector<double> scan_key, scan_key_pending;
  int64_t range_lo = -1, range_hi = -1;  // ctx_set_range: sub-batch of the next call (comm.cu)
  // Pinned staging for small transfers: the model upload of every call (F, G, dt, shared
  // parameters: a pageable source would make cudaMemcpyAsync stage it synchronously) goes through
  // a ring of pinned slots, and host-buffer calls whose arrays total <= kTinyBytes travel as ONE
  // H2D and ONE D2H copy through `bounce` instead of one copy per field.
  struct PinSlot { char *host = nullptr; cudaEvent_t done = nullptr; };
  PinSlot pin[4];
  int pin_next = 0;
  char *bounce = nullptr;
  char *pit_buf = nullptr;               // host-buffer staging of BDLM_PARALLEL_IN_TIME calls
  size_t pit_bytes = 0;
  ScanPeers scan_peers{};                // scan_set_peers: mailbox exchange of the dist scan phases
  const unsigned long long *scan_epoch = nullptr;
};

static std::string g_create_err;

// NVTX range around every ABI call and every slab phase of the host-buffer pipeline (SURVEY.md
// section 5, tracing row): shows up in Nsight Systems / ncu --nvtx as bdlm_* ranges.
struct NvtxRange {
  explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
  NvtxRange(const NvtxRange &) = delete;
  NvtxRange &operator=(const NvtxRange &) = delete;
};

namespace {

enum ApiOp { A_FILTER, A_SMOOTH, A_FILTER_SMOOTH, A_LOGLIK, A_FFBS, A_SVD_FILTER, A_SVD_FFBS,
             A_STATS,
             // "next" rows (SURVEY.md 8f)
             A_AR_FILTER, A_AR_FFBS, A_CONJ_FILTER, A_GIBBS_DRAW };

int fail(bdlm_ctx *c, int code, const std::string &msg) {
  if (c) c->err = msg; else g_create_err = msg;
  return code;
}

#define CU(call)                                                                        \
  do {                                                                                  \
    cudaError_t e_ = (call);                                                            \
    if (e_ != cudaSuccess)                                                              \
      return fail(c, BDLM_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));  \
  } while (0)

size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

constexpr size_t kPinSlotBytes = 64 << 10;   // model upload slots
constexpr size_t kTinyBytes = 512 << 10;     // host-buffer calls below this use the bounce path

// Host -> device copy of a small block the caller is about to free (std::vector): through a pinned
// slot when it fits (really asynchronous), else straight from pageable memory (the driver stages it
// before returning).
int upload_small(bdlm_ctx *c, void *dev, const void *host, size_t bytes) {
  if (bytes == 0) return 0;
  if (bytes <= kPinSlotBytes) {
    bdlm_ctx::PinSlot &sl = c->pin[c->pin_next];
    c->pin_next = (c->pin_next + 1) & 3;
    if (!sl.host) {
      CU(cudaHostAlloc(reinterpret_cast<void **>(&sl.host), kPinSlotBytes, cudaHostAllocDefault));
      CU(cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming));
    } else {
      CU(cudaEventSynchronize(sl.done));  // the copy that last used this slot has left it
    }
    std::memcpy(sl.host, host, bytes);
    CU(cudaMemcpyAsync(dev, sl.host, bytes, cudaMemcpyHostToDevice, c->stream));
    CU(cudaEventRecord(sl.done, c->stream));
    return 0;
  }
  CU(cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, c->stream));
  return 0;
}

int ensure_arena(bdlm_ctx *c, size_t bytes) {
  if (bytes <= c->arena_bytes) return 0;
  CU(cudaStreamSynchronize(c->stream));
  CU(cudaStreamSynchronize(c->s_in));
  CU(cudaStreamSynchronize(c->s_out));
  if (c->arena) CU(cudaFree(c->arena));
  c->arena = nullptr; c->arena_bytes = 0;
  CU(cudaMalloc(&c->arena, bytes));
  c->arena_bytes = bytes;
  return 0;
}

struct Bump {
  char *base; size_t off, cap;
  template <class T> T *take(size_t count) {
    off = align_up(off);
    T *p = reinterpret_cast<T *>(base + off);
    off += count * sizeof(T);
    return p;
  }
};

// One fully device-resident invocation over series [b0, b0 + Bc) of arrays whose batch
// pitch is Bp.
struct DevCall {
  int op;
  bdlm_problem pr;  // F, G, times: host; everything else device
  int64_t b0, Bc, Bp;
  int64_t rng_b0 = 0;  // index of series b0 within the CALL (slabs / chunks restart b0 at 0)
  bdlm_kf_out kf{};
  bdlm_smooth_out sm{};
  bdlm_svd_out svd{};
  bdlm_gibbs_stats stats{};
  const double *z = nullptr;
  double *theta = nullptr;
  double *ll_tr = nullptr, *ll_in = nullptr;
  int32_t *status = nullptr;
  // scalar AR(1) / OU calls: pr carries B, T, layout, mem, times, y with n = p = 1
  bdlm_ar_problem ar{};
  bdlm_ar_out ar_out{};
  // conjugate filter
  double cj_shape = 0, cj_scale = 0;
  double *cj_shape_out = nullptr, *cj_scale_out = nullptr;
  // last filtered state only (rides on the log-likelihood kernels)
  double *last_m = nullptr, *last_C = nullptr;
  // conjugate draws
  bdlm_gibbs_prior prior{};
  bdlm_gibbs_rng rng{};
  double *V_out = nullptr, *W_out = nullptr, *v_sr = nullptr, *w_sr = nullptr;
};

int rows_of(const bdlm_problem &p) { return p.T + (p.keep_init ? 1 : 0); }

View mk_view(double *ptr, int layout, int64_t b0, int64_t Bp, int64_t R, int64_t k) {
  View v{nullptr, 0, 0, 0};
  if (!ptr) return v;
  if (layout == BDLM_TIME_MAJOR) { v.ptr = ptr + b0; v.sb = 1; v.sk = Bp; v.sr = k * Bp; }
  else { v.ptr = ptr + b0 * R * k; v.sb = R * k; v.sr = k; v.sk = 1; }
  return v;
}
CView mk_cview(const double *ptr, int layout, int64_t b0, int64_t Bp, int64_t R, int64_t k) {
  View v = mk_view(const_cast<double *>(ptr), layout, b0, Bp, R, k);
  return CView{v.ptr, v.sb, v.sr, v.sk};
}
View mk_rowview(double *ptr, int layout, int64_t b0, int64_t Bp, int64_t k) {
  return mk_view(ptr, layout, b0, Bp, 1, k);  // one row per series
}

bool small_path(int op, const bdlm_problem &p) {
  return (op == A_FILTER || op == A_SMOOTH || op == A_FILTER_SMOOTH) && !p.v_tv && !p.w_tv &&
         small_supported(p.n, p.p);
}

int warp_op(int op) {
  switch (op) {
    case A_FILTER: return kOpFilter;
    case A_SMOOTH: return kOpSmooth;
    case A_FILTER_SMOOTH: return kOpFilterSmooth;
    case A_LOGLIK: return kOpLoglik;
    case A_FFBS: return kOpFfbs;
    case A_SVD_FILTER: return kOpSvdFilter;
    case A_SVD_FFBS: return kOpSvdFfbs;
    default: return kOpStats;
  }
}

// Per-series fields of a call, used for transposes (small path) and host staging.
struct Field {
  double **slot;  // address of the pointer inside the DevCall
  int64_t rows;   // rows per series (1 for per-series parameters / statistics)
  int64_t k;      // components per row
  bool in, out;
};

void collect_fields(DevCall &d, std::vector<Field> &f) {
  const bdlm_problem &p = d.pr;
  const int64_t n = p.n, pp = p.p, R = rows_of(p);
  auto add = [&](const double *const *slot, int64_t rows, int64_t k, bool in, bool out) {
    if (*slot) f.push_back(Field{const_cast<double **>(slot), rows, k, in, out});
  };
  if (d.op == A_AR_FILTER || d.op == A_AR_FFBS) {
    add(&d.pr.y, p.T, 1, true, false);
    if (d.ar.v_mode == BDLM_V_PER_SERIES_STEP) add(&d.ar.v, p.T, 1, true, false);
    if (d.ar.per_series) {
      add(&d.ar.phi, 1, 1, true, false);
      add(&d.ar.mu, 1, 1, true, false);
      add(&d.ar.sigma_eta, 1, 1, true, false);
    }
    add((const double *const *)&d.ar_out.m, R, 1, false, true);
    add((const double *const *)&d.ar_out.C, R, 1, false, true);
    add((const double *const *)&d.ar_out.a, R, 1, false, true);
    add((const double *const *)&d.ar_out.R, R, 1, false, true);
    add(&d.z, R, 1, true, false);
    add((const double *const *)&d.theta, R, 1, false, true);
    return;
  }
  if (d.op == A_GIBBS_DRAW) {
    add((const double *const *)&d.stats.ssy, 1, pp, true, false);
    add((const double *const *)&d.stats.ny, 1, pp, true, false);
    add((const double *const *)&d.stats.ssw, 1, n, true, false);
    add((const double *const *)&d.stats.scatter, 1, n * n, true, false);
    add(&d.rng.gamma_v, 1, pp, true, false);
    add(&d.rng.gamma_w, 1, n, true, false);
    add(&d.rng.bartlett, 1, n * n, true, false);
    add((const double *const *)&d.V_out, 1, pp * pp, false, true);
    add((const double *const *)&d.W_out, 1, n * n, false, true);
    add((const double *const *)&d.v_sr, 1, 2 * pp, false, true);
    add((const double *const *)&d.w_sr, 1, 2 * n, false, true);
    return;
  }
  const bool smooth_in = d.op == A_SMOOTH;
  if (d.op != A_SMOOTH) add(&d.pr.y, p.T, pp, true, false);
  // per-series time grids / model matrices travel (and are transposed / staged) like y
  if (p.per_series & BDLM_PS_TIMES) add(&d.pr.times, p.T, 1, true, false);
  if (p.per_series & BDLM_PS_F) add(&d.pr.F, p.T, n * pp, true, false);
  if (p.per_series & BDLM_PS_G) add(&d.pr.G, p.T, n * n, true, false);
  if (p.per_series & BDLM_PS_V) add(&d.pr.V, p.v_tv ? p.T : 1, pp * pp, true, false);
  if (p.per_series & BDLM_PS_W) add(&d.pr.W, p.w_tv ? p.T : 1, n * n, true, false);
  if (p.per_series & BDLM_PS_M0) add(&d.pr.m0, 1, n, true, false);
  if (p.per_series & BDLM_PS_C0) add(&d.pr.C0, 1, n * n, true, false);
  add((const double *const *)&d.kf.m, R, n, smooth_in, !smooth_in);
  add((const double *const *)&d.kf.C, R, n * n, smooth_in, !smooth_in);
  add((const double *const *)&d.kf.a, R, n, smooth_in, !smooth_in);
  add((const double *const *)&d.kf.R, R, n * n, smooth_in, !smooth_in);
  add((const double *const *)&d.kf.f, R, pp, false, true);
  add((const double *const *)&d.kf.Q, R, pp * pp, false, true);
  add((const double *const *)&d.sm.s, R, n, false, true);
  add((const double *const *)&d.sm.S, R, n * n, false, true);
  add((const double *const *)&d.svd.m, R, n, false, true);
  add((const double *const *)&d.svd.dc, R, n, false, true);
  add((const double *const *)&d.svd.uc, R, n * n, false, true);
  add((const double *const *)&d.svd.a, R, n, false, true);
  add((const double *const *)&d.svd.dr, R, n, false, true);
  add((const double *const *)&d.svd.ur, R, n * n, false, true);
  add((const double *const *)&d.svd.f, R, pp, false, true);
  add(&d.z, R, n, true, false);
  add((const double *const *)&d.theta, R, n, d.op == A_STATS, d.op != A_STATS);
  add((const double *const *)&d.stats.ssy, 1, pp, false, true);
  add((const double *const *)&d.stats.ny, 1, pp, false, true);
  add((const double *const *)&d.stats.ssw, 1, n, false, true);
  add((const double *const *)&d.stats.scatter, 1, n * n, false, true);
  add((const double *const *)&d.ll_tr, 1, 1, false, true);
  add((const double *const *)&d.ll_in, 1, 1, false, true);
  add((const double *const *)&d.last_m, 1, n, false, true);
  add((const double *const *)&d.last_C, 1, n * n, false, true);
  add((const double *const *)&d.cj_shape_out, R, 1, false, true);
  add((const double *const *)&d.cj_scale_out, R, 1, false, true);
}

// Device workspace (bytes) one run_dev call over Bc series needs beyond user arrays.
size_t dev_workspace_bytes(const DevCall &d, int64_t Bc) {
  const bdlm_problem &p = d.pr;
  const int64_t n = p.n, R = rows_of(p);
  size_t bytes = 0;
  // model: F, G, dt + shared params
  bytes += align_up(sizeof(double) * ((size_t)p.T * (n * p.p + n * n + 1) + 2 * n * n +
                                      (size_t)p.p * p.p * (p.v_tv ? p.T : 1) +
                                      (size_t)n * n * (p.w_tv ? p.T : 1) + n + 64)) + 4096;
  if (d.op == A_AR_FILTER || d.op == A_AR_FFBS) {
    bytes += align_up(sizeof(double) * 2 * (size_t)p.T);  // dt, shared v
    if (d.op == A_AR_FFBS) bytes += 2 * align_up(sizeof(double) * (size_t)R * Bc);  // (m, C) spill
    return bytes + 8192;
  }
  if (p.per_series & BDLM_PS_TIMES) bytes += align_up(sizeof(double) * (size_t)p.T * Bc);  // dt
  if (d.op == A_GIBBS_DRAW || d.op == A_CONJ_FILTER) return bytes + 8192;
  if (small_path(d.op, p)) {
    if (p.layout == BDLM_SERIES_MAJOR) {  // time-major mirrors of every field
      DevCall tmp = d;
      std::vector<Field> f;
      collect_fields(tmp, f);
      for (auto &x : f) bytes += align_up(sizeof(double) * (size_t)x.rows * x.k * Bc);
    }
    if (d.op == A_FILTER_SMOOTH) {
      if (!d.kf.m) bytes += align_up(sizeof(double) * (size_t)R * n * Bc);
      if (!d.kf.C) bytes += align_up(sizeof(double) * (size_t)R * n * n * Bc);
    }
  } else {
    bytes += align_up(sizeof(double) * warp_spill_doubles_per_row(warp_op(d.op), n, p.p) *
                      (size_t)R * Bc);
  }
  return bytes + 8192;
}

// Upload F, G, dt and shared parameters; fill the Batch description.
int upload_model(bdlm_ctx *c, const DevCall &d, Bump &bump, Batch &bt,
                 std::vector<double> &hG0, std::vector<double> &hF0) {
  const bdlm_problem &p = d.pr;
  const int n = p.n, pp = p.p, T = p.T;
  std::vector<double> host;
  auto push = [&](const double *src, size_t cnt) {
    size_t o = host.size();
    host.insert(host.end(), src, src + cnt);
    return o;
  };
  const bool psF = (p.per_series & BDLM_PS_F) != 0, psG = (p.per_series & BDLM_PS_G) != 0,
             psT = (p.per_series & BDLM_PS_TIMES) != 0;
  const size_t oF = psF ? 0 : push(p.F, (size_t)(p.f_tv ? T : 1) * n * pp);
  const size_t oG = psG ? 0 : push(p.G, (size_t)(p.g_tv ? T : 1) * n * n);
  // constant-bank copies of the first F, G for the register kernels (unused when they vary)
  if (psF) hF0.assign((size_t)n * pp, 0.0); else hF0.assign(p.F, p.F + (size_t)n * pp);
  if (psG) hG0.assign((size_t)n * n, 0.0); else hG0.assign(p.G, p.G + (size_t)n * n);
  size_t oDt = (size_t)-1;
  if (p.times && !psT) {
    double tmin = p.times[0];
    for (int t = 1; t < T; ++t) tmin = std::fmin(tmin, p.times[t]);
    // KalmanFilter.initialiseState, KalmanFilter.scala:116-117 -- or the time of a saved state
    double prev = p.t_init ? *p.t_init : tmin - 1.0;
    bool all_one = true;
    std::vector<double> dts(T);
    for (int t = 0; t < T; ++t) {
      dts[t] = p.times[t] - prev;
      prev = p.times[t];
      all_one = all_one && dts[t] == 1.0;
    }
    if (!all_one) oDt = push(dts.data(), T);
  }
  auto shared = [&](const double *src, int bit, size_t cnt) {
    return ((p.per_series & bit) || !src) ? (size_t)-1 : push(src, cnt);
  };
  const size_t oV = shared(p.V, BDLM_PS_V, (size_t)pp * pp * (p.v_tv ? T : 1));
  const size_t oW = shared(p.W, BDLM_PS_W, (size_t)n * n * (p.w_tv ? T : 1));
  const size_t oM = shared(p.m0, BDLM_PS_M0, n);
  const size_t oC = shared(p.C0, BDLM_PS_C0, (size_t)n * n);
  double *dev = bump.take<double>(host.size());
  {
    int rc = upload_small(c, dev, host.data(), host.size() * sizeof(double));
    if (rc) return rc;
  }
  bt.B = d.Bc; bt.T = T; bt.n = n; bt.p = pp; bt.keep_init = p.keep_init ? 1 : 0;
  bt.compat = p.compat;
  bt.f_tv = p.f_tv; bt.g_tv = p.g_tv;
  bt.ps_model = (psF || psG) ? 1 : 0;
  // per-step per-series array laid out like y with k components: strides of element (b, t, k)
  auto ps_strides = [&](const double *user, int64_t k, const double *&ptr, int64_t &sb, int64_t &sr,
                        int64_t &sk) {
    if (p.layout == BDLM_TIME_MAJOR) { ptr = user + d.b0; sb = 1; sk = d.Bp; sr = k * d.Bp; }
    else { ptr = user + d.b0 * (int64_t)T * k; sb = (int64_t)T * k; sr = k; sk = 1; }
  };
  if (psF) ps_strides(p.F, (int64_t)n * pp, bt.F, bt.F_sb, bt.F_sr, bt.F_sk);
  else { bt.F = dev + oF; bt.F_sb = 0; bt.F_sr = p.f_tv ? (int64_t)n * pp : 0; bt.F_sk = 1; }
  if (psG) ps_strides(p.G, (int64_t)n * n, bt.G, bt.G_sb, bt.G_sr, bt.G_sk);
  else { bt.G = dev + oG; bt.G_sb = 0; bt.G_sr = p.g_tv ? (int64_t)n * n : 0; bt.G_sk = 1; }
  bt.dt = (oDt == (size_t)-1) ? nullptr : dev + oDt;
  bt.dt_sb = 0; bt.dt_sr = 1;
  if (psT) {  // dt of every series on the device, in the layout of the times array
    const double *tp; int64_t tsb, tsr, tsk;
    ps_strides(p.times, 1, tp, tsb, tsr, tsk);
    double *dtw = bump.take<double>((size_t)T * d.Bc);
    if (p.layout == BDLM_TIME_MAJOR) { bt.dt_sb = 1; bt.dt_sr = d.Bc; }
    else { bt.dt_sb = T; bt.dt_sr = 1; }
    CU(launch_dt_from_times(tp, tsb, tsr, dtw, bt.dt_sb, bt.dt_sr, d.Bc, T, p.t_init, c->stream));
    ++c->launches;
    bt.dt = dtw;
  }
  auto pv = [&](const double *user, size_t off, int64_t k) {
    PView v{nullptr, 0, 1};
    if (off != (size_t)-1) { v.ptr = dev + off; v.sb = 0; v.sk = 1; }
    else if (!user) { /* not needed by this op */ }
    else if (p.layout == BDLM_TIME_MAJOR) { v.ptr = user + d.b0; v.sb = 1; v.sk = d.Bp; }
    else { v.ptr = user + d.b0 * k; v.sb = k; v.sk = 1; }
    return v;
  };
  bt.V = pv(p.V, oV, (int64_t)pp * pp);
  bt.v_tv = p.v_tv ? 1 : 0;
  bt.V_sr = 0;
  if (p.v_tv) {
    if (oV != (size_t)-1) bt.V_sr = (int64_t)pp * pp;  // shared: [T][p*p]
    else if (p.layout == BDLM_TIME_MAJOR) bt.V_sr = (int64_t)pp * pp * d.Bp;  // [T][k][B]
    else {  // [B][T][k]
      bt.V.ptr = p.V + d.b0 * (int64_t)T * pp * pp;
      bt.V.sb = (int64_t)T * pp * pp;
      bt.V_sr = (int64_t)pp * pp;
    }
  }
  bt.W = pv(p.W, oW, (int64_t)n * n);
  bt.w_tv = p.w_tv ? 1 : 0;
  bt.W_sr = 0;
  if (p.w_tv) {
    if (oW != (size_t)-1) bt.W_sr = (int64_t)n * n;  // shared: [T][n*n]
    else if (p.layout == BDLM_TIME_MAJOR) bt.W_sr = (int64_t)n * n * d.Bp;  // [T][k][B]
    else {  // [B][T][k]
      bt.W.ptr = p.W + d.b0 * (int64_t)T * n * n;
      bt.W.sb = (int64_t)T * n * n;
      bt.W_sr = (int64_t)n * n;
    }
  }
  bt.m0 = pv(p.m0, oM, n);
  bt.C0 = pv(p.C0, oC, (int64_t)n * n);
  bt.y = mk_cview(p.y, p.layout, d.b0, d.Bp, T, pp);
  bt.status = d.status ? d.status + d.b0 : nullptr;
  return 0;
}

// Run one device-resident call over [b0, b0 + Bc); workspace taken from `bump`.
int run_dev(bdlm_ctx *c, DevCall d, Bump bump) {
  const bdlm_problem &p = d.pr;
  const int64_t n = p.n, R = rows_of(p);
  Batch bt{};
  std::vector<double> hG0, hF0;

  if (d.op == A_AR_FILTER || d.op == A_AR_FFBS) {
    const bdlm_ar_problem &ap = d.ar;
    const int T = p.T, L = p.layout;
    ArArgs a{};
    a.B = d.Bc; a.T = T; a.ou = ap.process == BDLM_OU; a.ffbs = d.op == A_AR_FFBS;
    // host -> device: dt (OU; FilterOu.scala:35: t0 = head time, so dt[0] = 0) and shared v[T]
    std::vector<double> host;
    size_t oDt = (size_t)-1, oV = (size_t)-1;
    if (a.ou) {
      oDt = host.size();
      for (int t = 0; t < T; ++t)
        host.push_back(t == 0 ? 0.0 : (ap.times ? ap.times[t] - ap.times[t - 1] : 1.0));
    }
    if (ap.v_mode == BDLM_V_PER_STEP) { oV = host.size(); host.insert(host.end(), ap.v, ap.v + T); }
    if (!host.empty()) {
      double *dev = bump.take<double>(host.size());
      {
        int rc = upload_small(c, dev, host.data(), host.size() * sizeof(double));
        if (rc) return rc;
      }
      if (oDt != (size_t)-1) a.dt = dev + oDt;
      if (oV != (size_t)-1) a.v_shared = dev + oV;
    }
    auto row1 = [&](double *ptr, int64_t rows) {  // k = 1 view
      View v = mk_view(ptr, L, d.b0, d.Bp, rows, 1);
      return v;
    };
    auto par = [&](const double *ptr, double &scalar) {
      PView v{nullptr, 0, 1};
      if (ap.per_series) { v.ptr = ptr + d.b0; v.sb = 1; }
      else scalar = ptr[0];
      return v;
    };
    a.phi = par(ap.phi, a.phi_s); a.mu = par(ap.mu, a.mu_s); a.sigma = par(ap.sigma_eta, a.sigma_s);
    if (ap.v_mode == BDLM_V_SCALAR) a.v_s = ap.v[0];
    if (ap.v_mode == BDLM_V_PER_SERIES_STEP) a.v = row1(const_cast<double *>(ap.v), T);
    a.y = row1(const_cast<double *>(p.y), T);
    a.m = row1(d.ar_out.m, R); a.C = row1(d.ar_out.C, R);
    a.a = row1(d.ar_out.a, R); a.R = row1(d.ar_out.R, R);
    if (a.ffbs) {
      a.z = row1(const_cast<double *>(d.z), R);
      a.theta = row1(d.theta, R);
      // dense [R][Bc] workspace when the caller does not want (m, C)
      a.sm = d.ar_out.m ? a.m : mk_view(bump.take<double>((size_t)R * d.Bc), BDLM_TIME_MAJOR, 0, d.Bc, R, 1);
      a.sC = d.ar_out.C ? a.C : mk_view(bump.take<double>((size_t)R * d.Bc), BDLM_TIME_MAJOR, 0, d.Bc, R, 1);
    }
    CU(launch_ar(a, c->stream));
    ++c->launches;
    return 0;
  }

  if (d.op == A_GIBBS_DRAW) {
    const int L = p.layout;
    GibbsDrawArgs a{};
    a.B = d.Bc; a.n = p.n; a.p = p.p; a.T = p.T;
    a.wishart = d.prior.w_psi != nullptr;
    a.v_shape = d.prior.v_shape; a.v_scale = d.prior.v_scale;
    a.w_shape = d.prior.w_shape; a.w_scale = d.prior.w_scale; a.w_nu = d.prior.w_nu;
    if (a.wishart) {
      double *dev = bump.take<double>((size_t)n * n);
      CU(cudaMemcpyAsync(dev, d.prior.w_psi, sizeof(double) * n * n, cudaMemcpyHostToDevice, c->stream));
      a.psi = dev;
    }
    a.stats.ssy = mk_rowview(d.stats.ssy, L, d.b0, d.Bp, p.p);
    a.stats.ny = mk_rowview(d.stats.ny, L, d.b0, d.Bp, p.p);
    a.stats.ssw = mk_rowview(d.stats.ssw, L, d.b0, d.Bp, n);
    a.stats.scatter = mk_rowview(d.stats.scatter, L, d.b0, d.Bp, n * n);
    a.gv = mk_rowview(const_cast<double *>(d.rng.gamma_v), L, d.b0, d.Bp, p.p);
    a.gw = mk_rowview(const_cast<double *>(d.rng.gamma_w), L, d.b0, d.Bp, n);
    a.bart = mk_rowview(const_cast<double *>(d.rng.bartlett), L, d.b0, d.Bp, n * n);
    a.seed = d.rng.seed; a.sweep = d.rng.sweep; a.base = c->rng_first + d.rng_b0;
    a.V = mk_rowview(d.V_out, L, d.b0, d.Bp, (int64_t)p.p * p.p);
    a.W = mk_rowview(d.W_out, L, d.b0, d.Bp, n * n);
    a.v_shape_rate = mk_rowview(d.v_sr, L, d.b0, d.Bp, 2 * p.p);
    a.w_shape_rate = mk_rowview(d.w_sr, L, d.b0, d.Bp, 2 * n);
    a.status = d.status ? d.status + d.b0 : nullptr;
    if (a.status) CU(cudaMemsetAsync(a.status, 0, sizeof(int32_t) * d.Bc, c->stream));
    CU(launch_gibbs_draw(a, c->stream, &c->launches));
    return 0;
  }

  if (d.op == A_CONJ_FILTER) {
    int rc = upload_model(c, d, bump, bt, hG0, hF0);
    if (rc) return rc;
    const int L = p.layout;
    ConjArgs a{};
    a.bt = bt;
    a.prior_shape = d.cj_shape; a.prior_scale = d.cj_scale;
    a.kf.m = mk_view(d.kf.m, L, d.b0, d.Bp, R, n); a.kf.C = mk_view(d.kf.C, L, d.b0, d.Bp, R, n * n);
    a.kf.a = mk_view(d.kf.a, L, d.b0, d.Bp, R, n); a.kf.R = mk_view(d.kf.R, L, d.b0, d.Bp, R, n * n);
    a.kf.f = mk_view(d.kf.f, L, d.b0, d.Bp, R, 1); a.kf.Q = mk_view(d.kf.Q, L, d.b0, d.Bp, R, 1);
    a.shape = mk_view(d.cj_shape_out, L, d.b0, d.Bp, R, 1);
    a.scale = mk_view(d.cj_scale_out, L, d.b0, d.Bp, R, 1);
    if (bt.status) CU(cudaMemsetAsync(bt.status, 0, sizeof(int32_t) * d.Bc, c->stream));
    CU(launch_conjugate(a, hG0.data(), hF0.data(), c->stream));
    ++c->launches;
    return 0;
  }

  if (small_path(d.op, p)) {
    int layout = p.layout;
    std::vector<Field> fields;
    std::vector<double *> user_ptrs;
    if (layout == BDLM_SERIES_MAJOR) {
      // Mirror every per-series field in time-major workspace; transpose inputs in.
      collect_fields(d, fields);
      for (auto &f : fields) {
        double *user = *f.slot + d.b0 * f.rows * f.k;
        double *tm = bump.take<double>((size_t)f.rows * f.k * d.Bc);
        user_ptrs.push_back(user);
        if (f.in) {
          CU(launch_transpose(user, tm, d.Bc, f.rows * f.k, c->stream));
          ++c->launches;
        }
        *f.slot = tm;
      }
      if (d.status) d.status += d.b0;
      d.pr.layout = BDLM_TIME_MAJOR;
      d.b0 = 0; d.Bp = d.Bc;
    }
    int rc = upload_model(c, d, bump, bt, hG0, hF0);
    if (rc) return rc;
    auto uv = [&](double *ptr, int64_t k) {
      return mk_view(ptr, BDLM_TIME_MAJOR, d.b0, d.Bp, R, k);
    };
    KfViews kv;
    kv.m = uv(d.kf.m, n); kv.C = uv(d.kf.C, n * n);
    kv.a = uv(d.kf.a, n); kv.R = uv(d.kf.R, n * n);
    kv.f = uv(d.kf.f, p.p); kv.Q = uv(d.kf.Q, (int64_t)p.p * p.p);
    View sv = uv(d.sm.s, n), Sv = uv(d.sm.S, n * n);
    if (d.op == A_FILTER_SMOOTH) {
      // (m, C) spill for the backward pass when the caller does not want them: dense
      // [R][k][Bc] workspace (pitch Bc, offset 0), unlike user arrays (pitch Bp, offset b0)
      if (!d.kf.m)
        kv.m = mk_view(bump.take<double>((size_t)R * n * d.Bc), BDLM_TIME_MAJOR, 0, d.Bc, R, n);
      if (!d.kf.C)
        kv.C = mk_view(bump.take<double>((size_t)R * n * n * d.Bc), BDLM_TIME_MAJOR, 0, d.Bc, R,
                       n * n);
    }
    CU(launch_kf_small(bt, hG0.data(), hF0.data(), kv, sv, Sv, d.op != A_SMOOTH,
                       d.op != A_FILTER, c->stream));
    ++c->launches;
    if (layout == BDLM_SERIES_MAJOR) {
      for (size_t i = 0; i < fields.size(); ++i)
        if (fields[i].out) {
          CU(launch_transpose(*fields[i].slot, user_ptrs[i], fields[i].rows * fields[i].k,
                              d.Bc, c->stream));
          ++c->launches;
        }
    }
    return 0;
  }

  // ---- warp-per-series path ----
  int rc = upload_model(c, d, bump, bt, hG0, hF0);
  if (rc) return rc;
  if (d.op == A_FFBS && ffbs_small_supported(bt)) {
    // one thread per chain (ffbs_small.cu); (m, C) spill in the caller's arrays when they are
    // wanted, else dense time-major workspace
    const int L = p.layout;
    FfbsSmallArgs fa{};
    fa.bt = bt;
    fa.kf.a = mk_view(d.kf.a, L, d.b0, d.Bp, R, n); fa.kf.R = mk_view(d.kf.R, L, d.b0, d.Bp, R, n * n);
    fa.kf.f = mk_view(d.kf.f, L, d.b0, d.Bp, R, 1); fa.kf.Q = mk_view(d.kf.Q, L, d.b0, d.Bp, R, 1);
    fa.sm = d.kf.m ? mk_view(d.kf.m, L, d.b0, d.Bp, R, n)
                   : mk_view(bump.take<double>((size_t)R * n * d.Bc), BDLM_TIME_MAJOR, 0, d.Bc, R, n);
    fa.sC = d.kf.C ? mk_view(d.kf.C, L, d.b0, d.Bp, R, n * n)
                   : mk_view(bump.take<double>((size_t)R * n * n * d.Bc), BDLM_TIME_MAJOR, 0, d.Bc, R, n * n);
    fa.z = mk_cview(d.z, L, d.b0, d.Bp, R, n);
    fa.theta = mk_view(d.theta, L, d.b0, d.Bp, R, n);
    fa.stats.ssy = mk_rowview(d.stats.ssy, L, d.b0, d.Bp, 1);
    fa.stats.ny = mk_rowview(d.stats.ny, L, d.b0, d.Bp, 1);
    fa.stats.ssw = mk_rowview(d.stats.ssw, L, d.b0, d.Bp, n);
    fa.stats.scatter = mk_rowview(d.stats.scatter, L, d.b0, d.Bp, n * n);
    fa.rng_seed = c->rng_seed; fa.rng_sweep = c->rng_sweep; fa.rng_base = c->rng_first + d.rng_b0;
    CU(launch_ffbs_small(fa, hG0.data(), hF0.data(), c->stream));
    ++c->launches;
    return 0;
  }
  if (d.op == A_LOGLIK && loglik_small_supported(bt)) {
    // thread-per-series log-likelihoods (scalar_filters.cu): strided views serve both layouts
    CU(launch_loglik_small(bt, hG0.data(), hF0.data(), d.ll_tr ? d.ll_tr + d.b0 : nullptr,
                           d.ll_in ? d.ll_in + d.b0 : nullptr,
                           mk_rowview(d.last_m, p.layout, d.b0, d.Bp, n),
                           mk_rowview(d.last_C, p.layout, d.b0, d.Bp, n * n), c->stream));
    ++c->launches;
    return 0;
  }
  WarpArgs wa{};
  wa.bt = bt;
  const int L = p.layout;
  wa.kf.m = mk_view(d.kf.m, L, d.b0, d.Bp, R, n);
  wa.kf.C = mk_view(d.kf.C, L, d.b0, d.Bp, R, n * n);
  wa.kf.a = mk_view(d.kf.a, L, d.b0, d.Bp, R, n);
  wa.kf.R = mk_view(d.kf.R, L, d.b0, d.Bp, R, n * n);
  wa.kf.f = mk_view(d.kf.f, L, d.b0, d.Bp, R, p.p);
  wa.kf.Q = mk_view(d.kf.Q, L, d.b0, d.Bp, R, (int64_t)p.p * p.p);
  wa.s = mk_view(d.sm.s, L, d.b0, d.Bp, R, n);
  wa.S = mk_view(d.sm.S, L, d.b0, d.Bp, R, n * n);
  wa.z = mk_cview(d.z, L, d.b0, d.Bp, R, n);
  wa.rng_seed = c->rng_seed; wa.rng_sweep = c->rng_sweep;
  wa.rng_base = c->rng_first + d.rng_b0;
  wa.theta = mk_view(d.theta, L, d.b0, d.Bp, R, n);
  wa.svd.m = mk_view(d.svd.m, L, d.b0, d.Bp, R, n);
  wa.svd.dc = mk_view(d.svd.dc, L, d.b0, d.Bp, R, n);
  wa.svd.uc = mk_view(d.svd.uc, L, d.b0, d.Bp, R, n * n);
  wa.svd.a = mk_view(d.svd.a, L, d.b0, d.Bp, R, n);
  wa.svd.dr = mk_view(d.svd.dr, L, d.b0, d.Bp, R, n);
  wa.svd.ur = mk_view(d.svd.ur, L, d.b0, d.Bp, R, n * n);
  wa.svd.f = mk_view(d.svd.f, L, d.b0, d.Bp, R, p.p);
  wa.stats.ssy = mk_rowview(d.stats.ssy, L, d.b0, d.Bp, p.p);
  wa.stats.ny = mk_rowview(d.stats.ny, L, d.b0, d.Bp, p.p);
  wa.stats.ssw = mk_rowview(d.stats.ssw, L, d.b0, d.Bp, n);
  wa.stats.scatter = mk_rowview(d.stats.scatter, L, d.b0, d.Bp, n * n);
  wa.last_m = mk_rowview(d.last_m, L, d.b0, d.Bp, n);
  wa.last_C = mk_rowview(d.last_C, L, d.b0, d.Bp, n * n);
  wa.ll_transition = d.ll_tr ? d.ll_tr + d.b0 : nullptr;
  wa.ll_innov = d.ll_in ? d.ll_in + d.b0 : nullptr;
  const int wop = warp_op(d.op);
  wa.spill_k = (int64_t)warp_spill_doubles_per_row(wop, p.n, p.p);
  wa.spill = wa.spill_k ? bump.take<double>((size_t)wa.spill_k * R * d.Bc) : nullptr;
  if (!p.v_tv && !p.w_tv && !bt.ps_model && bt.dt_sb == 0 &&
      group_supported(wop, p.n, p.p, p.keep_init ? 1 : 0)) {
    CU(launch_group(wop, wa, c->stream));  // two series per warp, compile-time n (kf_group.cu)
    ++c->launches;
    return 0;
  }
  CU(launch_warp(wop, wa, c->stream));
  ++c->launches;
  return 0;
}

int validate(bdlm_ctx *c, int op, const bdlm_problem *p) {
  if (!c) return fail(nullptr, BDLM_E_ARG, "null context");
  if (!p) return fail(c, BDLM_E_ARG, "null problem");
  if (p->T == 0) return fail(c, BDLM_E_EMPTY, "T == 0: empty observation vector");
  if (p->B < 0 || p->T < 0) return fail(c, BDLM_E_ARG, "negative B or T");
  if (p->n < 1 || p->n > BDLM_MAX_N || p->p < 1 || p->p > BDLM_MAX_P)
    return fail(c, BDLM_E_ARG, "unsupported n (1..48) or p (1..32)");
  if (op != A_GIBBS_DRAW && op != A_AR_FILTER && op != A_AR_FFBS && op != A_CONJ_FILTER &&
      warp_smem_bytes(warp_op(op), p->n, p->p) > (size_t)227 * 1024)
    return fail(c, BDLM_E_ARG, "n and p together exceed one SM's shared memory (227 KB) for this "
                               "operation: reduce p (n = 48 runs with p <= 16 on the Kalman path, "
                               "p <= 8 on the SVD path)");
  if (p->layout != BDLM_TIME_MAJOR && p->layout != BDLM_SERIES_MAJOR)
    return fail(c, BDLM_E_ARG, "bad layout");
  if (p->mem != BDLM_DEVICE && p->mem != BDLM_HOST) return fail(c, BDLM_E_ARG, "bad mem");
  if (op != A_GIBBS_DRAW && (!p->F || !p->G)) return fail(c, BDLM_E_ARG, "null F or G");
  if (p->per_series & ~(BDLM_PS_V | BDLM_PS_W | BDLM_PS_M0 | BDLM_PS_C0 | BDLM_PS_TIMES | BDLM_PS_F |
                        BDLM_PS_G))
    return fail(c, BDLM_E_ARG, "unknown per_series bit");
  if ((p->per_series & BDLM_PS_TIMES) && !p->times)
    return fail(c, BDLM_E_ARG, "BDLM_PS_TIMES without a times array");
  if ((p->per_series & BDLM_PS_TIMES) && p->g_tv && !(p->per_series & BDLM_PS_G))
    return fail(c, BDLM_E_ARG, "per-series time grids with a dt-dependent G need per-series G "
                               "(BDLM_PS_G): g(dt) differs by series");
  if ((p->per_series & BDLM_PS_F) && !p->f_tv) return fail(c, BDLM_E_ARG, "BDLM_PS_F needs f_tv = 1");
  if ((p->per_series & BDLM_PS_G) && !p->g_tv) return fail(c, BDLM_E_ARG, "BDLM_PS_G needs g_tv = 1");
  if ((p->per_series & (BDLM_PS_TIMES | BDLM_PS_F | BDLM_PS_G)) &&
      (op == A_CONJ_FILTER || op == A_GIBBS_DRAW))
    return fail(c, BDLM_E_ARG, "per-series grids / models: not supported by this entry point");
  if (op == A_GIBBS_DRAW) return 0;
  if (op == A_CONJ_FILTER) {
    if (!p->W || !p->m0 || !p->C0 || !p->y) return fail(c, BDLM_E_ARG, "null W, m0, C0 or y");
    return 0;
  }
  if (op != A_STATS && (!p->V || !p->W)) return fail(c, BDLM_E_ARG, "null V or W");
  if (op != A_SMOOTH && op != A_STATS && (!p->m0 || !p->C0))
    return fail(c, BDLM_E_ARG, "null m0 or C0");
  if (op != A_SMOOTH && !p->y) return fail(c, BDLM_E_ARG, "null y");
  if (p->v_tv && op != A_FILTER && op != A_FILTER_SMOOTH && op != A_FFBS && op != A_LOGLIK &&
      op != A_SVD_FILTER && op != A_SVD_FFBS)
    return fail(c, BDLM_E_ARG, "v_tv: supported by filter, filter+smoother, log-likelihood, FFBS, "
                               "SVD filter and SVD FFBS");
  if (p->w_tv && op != A_FILTER && op != A_FILTER_SMOOTH && op != A_FFBS && op != A_SVD_FILTER &&
      op != A_SVD_FFBS)
    return fail(c, BDLM_E_ARG, "w_tv: supported by filter, filter+smoother, FFBS, SVD filter and "
                               "SVD FFBS");
  if ((op == A_FFBS || op == A_SVD_FFBS || op == A_STATS) && !p->keep_init)
    return fail(c, BDLM_E_ARG, "FFBS keeps the initial state: keep_init must be 1");
  return 0;
}

// Device-mode entry: loop over series chunks that fit the workspace cap.
int run_device_mode(bdlm_ctx *c, DevCall d, int64_t lo, int64_t hi) {
  const int64_t B = d.pr.B;
  if (hi <= lo) return 0;
  int64_t chunk = hi - lo;
  while (chunk > 128 && dev_workspace_bytes(d, chunk) > c->workspace_cap)
    chunk = ((chunk / 2 + 127) / 128) * 128;
  // series-major small path transposes are addressed per chunk; any chunk size works
  const size_t need = dev_workspace_bytes(d, chunk);
  int rc = ensure_arena(c, need);
  if (rc) return rc;
  for (int64_t b0 = lo; b0 < hi; b0 += chunk) {
    DevCall s = d;
    s.b0 = b0; s.Bc = std::min(chunk, hi - b0); s.Bp = B; s.rng_b0 = b0;
    Bump bump{c->arena, 0, c->arena_bytes};
    rc = run_dev(c, s, bump);
    if (rc) return rc;
  }
  return 0;
}

// Host-mode entry: stage slabs of series through the arena with two buffer sets so the
// H2D copy of slab i+1, the kernels of slab i and the D2H copy of slab i-1 overlap.
int run_host_mode(bdlm_ctx *c, DevCall d, int64_t lo, int64_t hi) {
  const bdlm_problem &p = d.pr;
  const int64_t B = p.B;
  if (hi <= lo) return 0;
  std::vector<Field> fields;
  collect_fields(d, fields);
  std::vector<double *> host_ptrs;
  for (auto &f : fields) host_ptrs.push_back(*f.slot);
  int32_t *host_status = d.status;
  size_t per_series = sizeof(int32_t);
  for (auto &f : fields) per_series += sizeof(double) * (size_t)f.rows * f.k;

  // ---- small calls (one series of T = 10 ... 1000, a few hundred short series): every field
  // packed into one pinned block, ONE copy in, ONE copy out, everything on the context's stream.
  // The per-field pipeline below costs one cudaMemcpyAsync (5-10 us from pageable memory) per
  // field and three streams' worth of events, which dominates calls of this size.
  if (lo == 0 && hi == B &&
      per_series * (size_t)B + 256 * (fields.size() + 2) <= std::min(kTinyBytes, c->staging_cap / 4)) {
    std::vector<size_t> off(fields.size());
    size_t in_end = 0, pos = 0;
    for (int pass = 0; pass < 2; ++pass) {  // inputs first, then outputs: two contiguous regions
      for (size_t i = 0; i < fields.size(); ++i) {
        if ((pass == 0) != fields[i].in) continue;
        off[i] = pos;
        pos = align_up(pos + sizeof(double) * (size_t)fields[i].rows * fields[i].k * B);
      }
      if (pass == 0) in_end = pos;
    }
    const size_t st_off = pos;
    pos = align_up(pos + sizeof(int32_t) * (size_t)B);
    const size_t staged = pos;
    DevCall t = d;
    t.pr.mem = BDLM_DEVICE;
    int rc = ensure_arena(c, staged + dev_workspace_bytes(t, B) + 65536);
    if (rc) return rc;
    if (!c->bounce) CU(cudaHostAlloc(reinterpret_cast<void **>(&c->bounce), 2 * kTinyBytes, cudaHostAllocDefault));
    CU(cudaStreamSynchronize(c->stream));  // earlier device-mode work may still use the arena / bounce
    for (size_t i = 0; i < fields.size(); ++i)
      if (fields[i].in)
        std::memcpy(c->bounce + off[i], host_ptrs[i], sizeof(double) * (size_t)fields[i].rows * fields[i].k * B);
    if (in_end) CU(cudaMemcpyAsync(c->arena, c->bounce, in_end, cudaMemcpyHostToDevice, c->stream));
    {
      std::vector<Field> tf;
      collect_fields(t, tf);
      for (size_t i = 0; i < tf.size(); ++i) *tf[i].slot = reinterpret_cast<double *>(c->arena + off[i]);
      t.status = host_status ? reinterpret_cast<int32_t *>(c->arena + st_off) : nullptr;
      t.b0 = 0; t.Bc = B; t.Bp = B; t.rng_b0 = 0;
      Bump work{c->arena, staged, c->arena_bytes};
      rc = run_dev(c, t, work);
      if (rc) return rc;
    }
    if (staged > in_end)
      CU(cudaMemcpyAsync(c->bounce + in_end, c->arena + in_end, staged - in_end, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    for (size_t i = 0; i < fields.size(); ++i)
      if (fields[i].out)
        std::memcpy(host_ptrs[i], c->bounce + off[i], sizeof(double) * (size_t)fields[i].rows * fields[i].k * B);
    if (host_status) std::memcpy(host_status, c->bounce + st_off, sizeof(int32_t) * (size_t)B);
    return 0;
  }

  // slab size: two staged sets + one device workspace within the staging cap
  int64_t slab = std::min<int64_t>(hi - lo, 1 << 20);
  auto total_for = [&](int64_t s) {
    DevCall t = d; t.pr.mem = BDLM_DEVICE;
    size_t staged = 0;
    for (auto &f : fields) staged += align_up(sizeof(double) * (size_t)f.rows * f.k * s);
    staged += align_up(sizeof(int32_t) * s);
    return 2 * staged + dev_workspace_bytes(t, s) + 65536;
  };
  while (slab > 128 && total_for(slab) > c->staging_cap) slab = ((slab / 2 + 127) / 128) * 128;
  int rc = ensure_arena(c, total_for(slab));
  if (rc) return rc;
  // Device-mode calls return without synchronising and use the same arena (spill, transposes,
  // model upload): the staged copies below run on other streams, so earlier work on the
  // context's stream must have drained before the first of them touches the arena.
  CU(cudaStreamSynchronize(c->stream));

  Bump bump{c->arena, 0, c->arena_bytes};
  std::vector<double *> dev_ptrs[2];
  int32_t *dev_status[2];
  for (int s = 0; s < 2; ++s) {
    for (auto &f : fields) dev_ptrs[s].push_back(bump.take<double>((size_t)f.rows * f.k * slab));
    dev_status[s] = bump.take<int32_t>(slab);
  }
  const Bump work = bump;

  auto copy = [&](const Field &f, double *host, double *dev, int64_t b0, int64_t Bs,
                  bool to_dev, cudaStream_t st) -> cudaError_t {
    const size_t rk = (size_t)f.rows * f.k;
    if (p.layout == BDLM_SERIES_MAJOR) {
      double *h = host + (size_t)b0 * rk;
      return to_dev ? cudaMemcpyAsync(dev, h, rk * Bs * sizeof(double), cudaMemcpyHostToDevice, st)
                    : cudaMemcpyAsync(h, dev, rk * Bs * sizeof(double), cudaMemcpyDeviceToHost, st);
    }
    double *h = host + b0;  // [rows*k][B] -> dense [rows*k][Bs]
    return to_dev ? cudaMemcpy2DAsync(dev, Bs * sizeof(double), h, B * sizeof(double),
                                      Bs * sizeof(double), rk, cudaMemcpyHostToDevice, st)
                  : cudaMemcpy2DAsync(h, B * sizeof(double), dev, Bs * sizeof(double),
                                      Bs * sizeof(double), rk, cudaMemcpyDeviceToHost, st);
  };

  int it = 0;
  for (int64_t b0 = lo; b0 < hi; b0 += slab, ++it) {
    const int s = it & 1;
    const int64_t Bs = std::min(slab, hi - b0);
    // the set's buffers are free once the D2H of the slab that used them has finished
    if (it >= 2) CU(cudaStreamWaitEvent(c->s_in, c->ev_out[s], 0));
    {
      NvtxRange r_("bdlm slab H2D");
      for (size_t i = 0; i < fields.size(); ++i)
        if (fields[i].in) CU(copy(fields[i], host_ptrs[i], dev_ptrs[s][i], b0, Bs, true, c->s_in));
    }
    CU(cudaEventRecord(c->ev_in[s], c->s_in));
    CU(cudaStreamWaitEvent(c->stream, c->ev_in[s], 0));
    if (it >= 2) CU(cudaStreamWaitEvent(c->stream, c->ev_out[s], 0));
    DevCall t = d;
    t.pr.mem = BDLM_DEVICE; t.pr.B = Bs; t.b0 = 0; t.Bc = Bs; t.Bp = Bs; t.rng_b0 = b0;
    {
      std::vector<Field> tf;
      collect_fields(t, tf);
      for (size_t i = 0; i < tf.size(); ++i) *tf[i].slot = dev_ptrs[s][i];
      t.status = host_status ? dev_status[s] : nullptr;
      NvtxRange r_("bdlm slab kernels");
      rc = run_dev(c, t, work);
      if (rc) return rc;
    }
    CU(cudaEventRecord(c->ev_comp[s], c->stream));
    CU(cudaStreamWaitEvent(c->s_out, c->ev_comp[s], 0));
    NvtxRange r_("bdlm slab D2H");
    for (size_t i = 0; i < fields.size(); ++i)
      if (fields[i].out) CU(copy(fields[i], host_ptrs[i], dev_ptrs[s][i], b0, Bs, false, c->s_out));
    if (host_status)
      CU(cudaMemcpyAsync(host_status + b0, dev_status[s], Bs * sizeof(int32_t),
                         cudaMemcpyDeviceToHost, c->s_out));
    CU(cudaEventRecord(c->ev_out[s], c->s_out));
  }
  CU(cudaStreamSynchronize(c->s_out));
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}

int dispatch(bdlm_ctx *c, DevCall &d) {
  CU(cudaSetDevice(c->device));
  d.b0 = 0; d.Bc = d.pr.B; d.Bp = d.pr.B;
  int64_t lo = 0, hi = d.pr.B;
  if (c->range_lo >= 0) {  // one shard of a batch cut over several contexts (comm.cu)
    lo = std::min(c->range_lo, d.pr.B); hi = std::min(c->range_hi, d.pr.B);
    c->range_lo = c->range_hi = -1;
  }
  return d.pr.mem == BDLM_HOST ? run_host_mode(c, d, lo, hi) : run_device_mode(c, d, lo, hi);
}

}  // namespace

namespace bdlm {
cudaStream_t ctx_stream(bdlm_ctx *c) { return c->stream; }
void ctx_set_range(bdlm_ctx *c, int64_t lo, int64_t hi) { c->range_lo = lo; c->range_hi = lo < 0 ? -1 : hi; }
void ctx_count_launches(bdlm_ctx *c, int64_t n) { c->launches += n; }
void scan_set_peers(bdlm_ctx *c, const ScanPeers *peers, const unsigned long long *epoch_dev) {
  if (peers) c->scan_peers = *peers; else c->scan_peers.world = 0;
  c->scan_epoch = epoch_dev;
}
}  // namespace bdlm

// ------------------------------------------------------------------------- C ABI

extern "C" {

int bdlm_version(void) { return BDLM_VERSION; }

int bdlm_create(int device, bdlm_ctx **out) {
  bdlm_ctx *c = nullptr;
  if (!out) return fail(nullptr, BDLM_E_ARG, "null out pointer");
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return fail(nullptr, BDLM_E_NODEVICE,
                std::string("no CUDA device (there is no CPU fallback): ") +
                    (e != cudaSuccess ? cudaGetErrorString(e) : "device count 0"));
  if (device < 0 || device >= count) return fail(nullptr, BDLM_E_ARG, "bad device index");
  e = cudaSetDevice(device);
  if (e != cudaSuccess) return fail(nullptr, BDLM_E_CUDA, cudaGetErrorString(e));
  c = new (std::nothrow) bdlm_ctx();
  if (!c) return fail(nullptr, BDLM_E_ARG, "out of host memory");
  c->device = device;
  bool ok = cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) == cudaSuccess &&
            cudaStreamCreateWithFlags(&c->s_in, cudaStreamNonBlocking) == cudaSuccess &&
            cudaStreamCreateWithFlags(&c->s_out, cudaStreamNonBlocking) == cudaSuccess;
  for (int i = 0; i < 2 && ok; ++i)
    ok = cudaEventCreateWithFlags(&c->ev_in[i], cudaEventDisableTiming) == cudaSuccess &&
         cudaEventCreateWithFlags(&c->ev_comp[i], cudaEventDisableTiming) == cudaSuccess &&
         cudaEventCreateWithFlags(&c->ev_out[i], cudaEventDisableTiming) == cudaSuccess;
  if (!ok) {
    g_create_err = std::string("stream/event creation failed: ") +
                   cudaGetErrorString(cudaGetLastError());
    bdlm_destroy(c);
    return BDLM_E_CUDA;
  }
  c->stream = c->own_stream;
  *out = c;
  return 0;
}

void bdlm_destroy(bdlm_ctx *c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  if (c->arena) cudaFree(c->arena);
  if (c->scan_table) cudaFree(c->scan_table);
  if (c->bounce) cudaFreeHost(c->bounce);
  if (c->pit_buf) cudaFree(c->pit_buf);
  for (auto &sl : c->pin) {
    if (sl.host) cudaFreeHost(sl.host);
    if (sl.done) cudaEventDestroy(sl.done);
  }
  for (int i = 0; i < 2; ++i) {
    if (c->ev_in[i]) cudaEventDestroy(c->ev_in[i]);
    if (c->ev_comp[i]) cudaEventDestroy(c->ev_comp[i]);
    if (c->ev_out[i]) cudaEventDestroy(c->ev_out[i]);
  }
  if (c->own_stream) cudaStreamDestroy(c->own_stream);
  if (c->s_in) cudaStreamDestroy(c->s_in);
  if (c->s_out) cudaStreamDestroy(c->s_out);
  delete c;
}

const char *bdlm_last_error(bdlm_ctx *c) { return c ? c->err.c_str() : g_create_err.c_str(); }

int bdlm_set_stream(bdlm_ctx *c, void *s, int use_own) {
  if (!c) return BDLM_E_ARG;
  cudaStream_t ns = use_own ? c->own_stream : reinterpret_cast<cudaStream_t>(s);
  if (ns != c->stream) c->scan_key.clear();  // the table upload was ordered on the old stream
  c->stream = ns;
  return 0;
}

int bdlm_set_rng(bdlm_ctx *c, uint64_t seed, uint64_t sweep, int64_t first_series) {
  if (!c) return BDLM_E_ARG;
  c->rng_seed = seed; c->rng_sweep = sweep; c->rng_first = first_series;
  return 0;
}

int bdlm_sync(bdlm_ctx *c) {
  if (!c) return BDLM_E_ARG;
  CU(cudaSetDevice(c->device));
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}

int64_t bdlm_launch_count(bdlm_ctx *c) { return c ? c->launches : 0; }

int64_t bdlm_wave_series(bdlm_ctx *c, int32_t n, int32_t p) {
  if (!c) return BDLM_E_ARG;
  if (!small_supported(n, p)) return fail(c, BDLM_E_ARG, "wave query: warp-kernel dimensions");
  CU(cudaSetDevice(c->device));
  Batch bt{};
  bt.n = n; bt.p = p;
  KfViews kv{};
  View v{nullptr, 0, 0, 0};
  int wave = 0;
  CU(launch_kf_small(bt, nullptr, nullptr, kv, v, v, true, true, c->stream, &wave));
  return wave;
}

int bdlm_fp64_peak_tflops(bdlm_ctx *c, double *tflops) {
  if (!c || !tflops) return BDLM_E_ARG;
  CU(cudaSetDevice(c->device));
  int rc = ensure_arena(c, 4096);
  if (rc) return rc;
  CU(measure_fp64_peak(c->stream, reinterpret_cast<double *>(c->arena), tflops));
  c->launches += 4;
  return 0;
}

int bdlm_set_staging_bytes(bdlm_ctx *c, int64_t bytes) {
  if (!c || bytes < ((int64_t)1 << 20)) return BDLM_E_ARG;
  c->staging_cap = (size_t)bytes;
  c->workspace_cap = std::max(c->workspace_cap, (size_t)bytes);
  return 0;
}

int bdlm_kf_filter(bdlm_ctx *c, const bdlm_problem *p, const bdlm_kf_out *out,
                   int32_t *status) {
  NvtxRange nvtx_("bdlm_kf_filter");
  int rc = validate(c, A_FILTER, p);
  if (rc) return rc;
  if (!out) return fail(c, BDLM_E_ARG, "null output struct");
  DevCall d{}; d.op = A_FILTER; d.pr = *p; d.kf = *out; d.status = status;
  return dispatch(c, d);
}

int bdlm_rts_smooth(bdlm_ctx *c, const bdlm_problem *p, const bdlm_kf_out *filt,
                    const bdlm_smooth_out *out, int32_t *status) {
  NvtxRange nvtx_("bdlm_rts_smooth");
  int rc = validate(c, A_SMOOTH, p);
  if (rc) return rc;
  if (!filt || !out || !filt->m || !filt->C)
    return fail(c, BDLM_E_ARG, "smoother needs filtered m and C");
  if (!out->s && !out->S) return fail(c, BDLM_E_ARG, "no smoother output requested");
  DevCall d{}; d.op = A_SMOOTH; d.pr = *p; d.kf = *filt; d.kf.f = nullptr; d.kf.Q = nullptr;
  d.sm = *out; d.status = status;
  return dispatch(c, d);
}

// BDLM_PARALLEL_IN_TIME: one long eligible series goes to the associative-scan kernels.  The
// forward pass alone (log-likelihoods, last state) runs any n <= 4; the smoother needs n = 1 or the
// textbook smoother, which is what its backward sweep computes.
static bool pit_eligible_forward(const bdlm_problem *p) {
  return (p->compat & BDLM_PARALLEL_IN_TIME) && p->B == 1 && p->T >= 4096 && p->p == 1 && p->n <= 4 &&
         !p->times && !p->f_tv && !p->g_tv && !p->per_series && !p->v_tv && !p->w_tv;
}
static bool pit_eligible(const bdlm_problem *p) {
  return pit_eligible_forward(p) && (p->n == 1 || (p->compat & BDLM_TEXTBOOK_SMOOTHER));
}

// Staging buffer of the host-buffer BDLM_PARALLEL_IN_TIME calls (the scan owns the arena); y is
// copied to its start.
static int pit_stage_y(bdlm_ctx *c, const bdlm_problem *p, size_t bytes) {
  CU(cudaSetDevice(c->device));
  if (bytes > c->pit_bytes) {
    CU(cudaStreamSynchronize(c->stream));
    if (c->pit_buf) CU(cudaFree(c->pit_buf));
    c->pit_buf = nullptr; c->pit_bytes = 0;
    CU(cudaMalloc(&c->pit_buf, bytes));
    c->pit_bytes = bytes;
  }
  CU(cudaMemcpyAsync(c->pit_buf, p->y, sizeof(double) * (size_t)p->T, cudaMemcpyHostToDevice, c->stream));
  return 0;
}

static int pit_host(bdlm_ctx *c, const bdlm_problem *p, const bdlm_kf_out *kf,
                    const bdlm_smooth_out *sm, int32_t *status) {
  // stage y in, every requested field out, through a buffer of its own (the scan owns the arena)
  const int64_t n = p->n, R = rows_of(*p);
  const int64_t ks[8] = {n, n * n, n, n * n, 1, 1, n, n * n};
  double *host[8] = {kf ? kf->m : nullptr, kf ? kf->C : nullptr, kf ? kf->a : nullptr, kf ? kf->R : nullptr,
                     kf ? kf->f : nullptr, kf ? kf->Q : nullptr, sm->s, sm->S};
  size_t off[9], pos = align_up(sizeof(double) * (size_t)p->T);
  for (int i = 0; i < 8; ++i) { off[i] = pos; if (host[i]) pos = align_up(pos + sizeof(double) * (size_t)R * ks[i]); }
  off[8] = pos; pos += 256;
  int rc0 = pit_stage_y(c, p, pos);
  if (rc0) return rc0;
  bdlm_problem q = *p;
  q.mem = BDLM_DEVICE;
  q.y = reinterpret_cast<const double *>(c->pit_buf);
  double *dev[8];
  for (int i = 0; i < 8; ++i) dev[i] = host[i] ? reinterpret_cast<double *>(c->pit_buf + off[i]) : nullptr;
  bdlm_kf_out dk = {dev[0], dev[1], dev[2], dev[3], dev[4], dev[5]};
  bdlm_smooth_out ds = {dev[6], dev[7]};
  int32_t *dst = status ? reinterpret_cast<int32_t *>(c->pit_buf + off[8]) : nullptr;
  int rc = bdlm_scan_filter_smooth(c, &q, &dk, &ds, dst);
  if (rc) return rc;
  for (int i = 0; i < 8; ++i)
    if (host[i])
      CU(cudaMemcpyAsync(host[i], dev[i], sizeof(double) * (size_t)R * ks[i], cudaMemcpyDeviceToHost, c->stream));
  if (status) CU(cudaMemcpyAsync(status, dst, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}

int bdlm_kf_filter_smooth(bdlm_ctx *c, const bdlm_problem *p, const bdlm_kf_out *kf,
                          const bdlm_smooth_out *sm, int32_t *status) {
  NvtxRange nvtx_("bdlm_kf_filter_smooth");
  int rc = validate(c, A_FILTER_SMOOTH, p);
  if (rc) return rc;
  if (!sm) return fail(c, BDLM_E_ARG, "null smoother output struct");
  if (pit_eligible(p) && (sm->s || sm->S)) {
    bdlm_problem q = *p;
    q.compat &= ~BDLM_PARALLEL_IN_TIME;
    return p->mem == BDLM_DEVICE ? bdlm_scan_filter_smooth(c, &q, kf, sm, status)
                                 : pit_host(c, &q, kf, sm, status);
  }
  DevCall d{}; d.op = A_FILTER_SMOOTH; d.pr = *p; if (kf) d.kf = *kf; d.sm = *sm;
  d.status = status;
  return dispatch(c, d);
}

// BDLM_PARALLEL_IN_TIME on bdlm_loglik / bdlm_kf_filter_last: bdlm_scan_loglik, with host buffers
// staged through pit_buf ([y | m_last | C_last | transition | innovations | status]).
static int pit_loglik(bdlm_ctx *c, const bdlm_problem *p, double *m_last, double *C_last,
                      double *transition, double *innovations, int32_t *status) {
  bdlm_problem q = *p;
  q.compat &= ~BDLM_PARALLEL_IN_TIME;
  if (p->mem == BDLM_DEVICE) return bdlm_scan_loglik(c, &q, m_last, C_last, transition, innovations, status);
  const int64_t n = p->n;
  const int64_t ks[4] = {n, n * n, 1, 1};
  double *host[4] = {m_last, C_last, transition, innovations};
  size_t off[5], pos = align_up(sizeof(double) * (size_t)p->T);
  for (int i = 0; i < 4; ++i) { off[i] = pos; if (host[i]) pos = align_up(pos + sizeof(double) * (size_t)ks[i]); }
  off[4] = pos; pos += 256;
  int rc = pit_stage_y(c, p, pos);
  if (rc) return rc;
  q.mem = BDLM_DEVICE;
  q.y = reinterpret_cast<const double *>(c->pit_buf);
  double *dev[4];
  for (int i = 0; i < 4; ++i) dev[i] = host[i] ? reinterpret_cast<double *>(c->pit_buf + off[i]) : nullptr;
  int32_t *dst = status ? reinterpret_cast<int32_t *>(c->pit_buf + off[4]) : nullptr;
  rc = bdlm_scan_loglik(c, &q, dev[0], dev[1], dev[2], dev[3], dst);
  if (rc) return rc;
  for (int i = 0; i < 4; ++i)
    if (host[i])
      CU(cudaMemcpyAsync(host[i], dev[i], sizeof(double) * (size_t)ks[i], cudaMemcpyDeviceToHost, c->stream));
  if (status) CU(cudaMemcpyAsync(status, dst, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}

int bdlm_loglik(bdlm_ctx *c, const bdlm_problem *p, double *transition, double *innovations,
                int32_t *status) {
  NvtxRange nvtx_("bdlm_loglik");
  int rc = validate(c, A_LOGLIK, p);
  if (rc) return rc;
  if (!transition && !innovations) return fail(c, BDLM_E_ARG, "no log-likelihood requested");
  if (pit_eligible_forward(p)) return pit_loglik(c, p, nullptr, nullptr, transition, innovations, status);
  DevCall d{}; d.op = A_LOGLIK; d.pr = *p; d.pr.keep_init = 1;
  d.ll_tr = transition; d.ll_in = innovations; d.status = status;
  return dispatch(c, d);
}

int bdlm_kf_filter_last(bdlm_ctx *c, const bdlm_problem *p, double *m_last, double *C_last,
                        double *transition, double *innovations, int32_t *status) {
  NvtxRange nvtx_("bdlm_kf_filter_last");
  int rc = validate(c, A_LOGLIK, p);
  if (rc) return rc;
  if (!m_last && !C_last && !transition && !innovations)
    return fail(c, BDLM_E_ARG, "nothing requested");
  if (pit_eligible_forward(p)) return pit_loglik(c, p, m_last, C_last, transition, innovations, status);
  DevCall d{}; d.op = A_LOGLIK; d.pr = *p; d.pr.keep_init = 1;
  d.last_m = m_last; d.last_C = C_last;
  d.ll_tr = transition; d.ll_in = innovations; d.status = status;
  return dispatch(c, d);
}

// BDLM_PARALLEL_IN_TIME on bdlm_ffbs: bdlm_scan_ffbs, with host buffers staged through pit_buf
// ([y | z | theta | m | C | a | R | f | Q | ssy | ny | ssw | scatter | status]).
static int pit_ffbs(bdlm_ctx *c, const bdlm_problem *p, const double *z, double *theta,
                    const bdlm_kf_out *kf, const bdlm_gibbs_stats *stats, int32_t *status) {
  bdlm_problem q = *p;
  q.compat &= ~BDLM_PARALLEL_IN_TIME;
  if (p->mem == BDLM_DEVICE) return bdlm_scan_ffbs(c, &q, z, theta, kf, stats, status);
  const int64_t n = p->n, R = rows_of(*p);
  // outputs: theta, kf fields, statistics (rows x k, or k for a statistic)
  const int64_t ks[11] = {R * n, R * n, R * n * n, R * n, R * n * n, R, R, 1, 1, n, n * n};
  double *host[11] = {theta,
                      kf ? kf->m : nullptr, kf ? kf->C : nullptr, kf ? kf->a : nullptr, kf ? kf->R : nullptr,
                      kf ? kf->f : nullptr, kf ? kf->Q : nullptr,
                      stats ? stats->ssy : nullptr, stats ? stats->ny : nullptr,
                      stats ? stats->ssw : nullptr, stats ? stats->scatter : nullptr};
  size_t pos = align_up(sizeof(double) * (size_t)p->T);
  const size_t z_off = pos;
  if (z) pos = align_up(pos + sizeof(double) * (size_t)(R * n));
  size_t off[12];
  for (int i = 0; i < 11; ++i) { off[i] = pos; if (host[i]) pos = align_up(pos + sizeof(double) * (size_t)ks[i]); }
  off[11] = pos; pos += 256;
  int rc = pit_stage_y(c, p, pos);
  if (rc) return rc;
  if (z) CU(cudaMemcpyAsync(c->pit_buf + z_off, z, sizeof(double) * (size_t)(R * n), cudaMemcpyHostToDevice,
                            c->stream));
  q.mem = BDLM_DEVICE;
  q.y = reinterpret_cast<const double *>(c->pit_buf);
  double *dev[11];
  for (int i = 0; i < 11; ++i) dev[i] = host[i] ? reinterpret_cast<double *>(c->pit_buf + off[i]) : nullptr;
  bdlm_kf_out dk = {dev[1], dev[2], dev[3], dev[4], dev[5], dev[6]};
  bdlm_gibbs_stats ds = {dev[7], dev[8], dev[9], dev[10]};
  int32_t *dst = status ? reinterpret_cast<int32_t *>(c->pit_buf + off[11]) : nullptr;
  rc = bdlm_scan_ffbs(c, &q, z ? reinterpret_cast<const double *>(c->pit_buf + z_off) : nullptr, dev[0],
                      kf ? &dk : nullptr, stats ? &ds : nullptr, dst);
  if (rc) return rc;
  for (int i = 0; i < 11; ++i)
    if (host[i])
      CU(cudaMemcpyAsync(host[i], dev[i], sizeof(double) * (size_t)ks[i], cudaMemcpyDeviceToHost, c->stream));
  if (status) CU(cudaMemcpyAsync(status, dst, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}

int bdlm_ffbs(bdlm_ctx *c, const bdlm_problem *p, const double *z, double *theta,
              const bdlm_kf_out *kf, const bdlm_gibbs_stats *stats, int32_t *status) {
  NvtxRange nvtx_("bdlm_ffbs");
  int rc = validate(c, A_FFBS, p);
  if (rc) return rc;
  if (!theta) return fail(c, BDLM_E_ARG, "null theta");  // z == NULL: on-device Philox normals
  if (pit_eligible_forward(p) && p->keep_init) return pit_ffbs(c, p, z, theta, kf, stats, status);
  DevCall d{}; d.op = A_FFBS; d.pr = *p; d.z = z; d.theta = theta;
  if (kf) d.kf = *kf;
  if (stats) d.stats = *stats;
  d.status = status;
  return dispatch(c, d);
}

int bdlm_svd_filter(bdlm_ctx *c, const bdlm_problem *p, const bdlm_svd_out *out,
                    int32_t *status) {
  NvtxRange nvtx_("bdlm_svd_filter");
  int rc = validate(c, A_SVD_FILTER, p);
  if (rc) return rc;
  if (!out) return fail(c, BDLM_E_ARG, "null output struct");
  DevCall d{}; d.op = A_SVD_FILTER; d.pr = *p; d.svd = *out; d.status = status;
  return dispatch(c, d);
}

int bdlm_svd_ffbs(bdlm_ctx *c, const bdlm_problem *p, const double *z, double *theta,
                  const bdlm_svd_out *filt, const bdlm_gibbs_stats *stats, int32_t *status) {
  NvtxRange nvtx_("bdlm_svd_ffbs");
  int rc = validate(c, A_SVD_FFBS, p);
  if (rc) return rc;
  if (!theta) return fail(c, BDLM_E_ARG, "null theta");  // z == NULL: on-device Philox normals
  DevCall d{}; d.op = A_SVD_FFBS; d.pr = *p; d.z = z; d.theta = theta;
  if (filt) d.svd = *filt;
  if (stats) d.stats = *stats;
  d.status = status;
  return dispatch(c, d);
}

// ---- parallel-in-time scan (scan.cu) ----------------------------------------------------

static int scan_validate(bdlm_ctx *c, const bdlm_problem *p) {
  int rc = validate(c, A_FILTER, p);
  if (rc) return rc;
  if (p->B != 1 || p->p != 1 || p->n > 4 || p->times || p->f_tv || p->g_tv || p->per_series ||
      p->mem != BDLM_DEVICE)
    return fail(c, BDLM_E_ARG,
                "scan path: B = 1, p = 1, n <= 4, regular grid, time-invariant model, shared "
                "parameters, device memory");
  return 0;
}

static int scan_fill(bdlm_ctx *c, const bdlm_problem *p, ScanArgs &a, bool forward = false) {
  a = ScanArgs{};
  a.n = p->n; a.T = p->T; a.keep_init = p->keep_init ? 1 : 0;
  a.G = p->G; a.F = p->F; a.W = p->W; a.V = p->V[0]; a.y = p->y;
  if (!forward) return 0;
  // The forward level-1 table depends on the model only: rebuild it when (n, G, F, W, V) change.
  if (!c->scan_table) CU(cudaMalloc(&c->scan_table, scan_table_bytes()));
  const int n = p->n;
  std::vector<double> key;
  key.push_back(n);
  key.insert(key.end(), p->G, p->G + n * n);
  key.insert(key.end(), p->F, p->F + n);
  key.insert(key.end(), p->W, p->W + n * n);
  key.push_back(p->V[0]);
  a.table = c->scan_table;
  a.table_upload = (key.size() != c->scan_key.size() ||
                    std::memcmp(key.data(), c->scan_key.data(), key.size() * sizeof(double)) != 0);
  if (a.table_upload) { c->scan_key.clear(); c->scan_key_pending = key; }
  return 0;
}

// launch_scan for a forward pass: the table key is committed only once the upload is enqueued, so
// a failed launch (or a finish phase without its local phase) can never leave a stale table that
// a later call would trust.
static int scan_launch_fwd(bdlm_ctx *c, ScanArgs &a, const ScanLoglikOut *ll = nullptr,
                           const ScanFfbsOut *fb = nullptr) {
  CU(ll   ? launch_scan_loglik(a, *ll, c->stream, &c->launches)
     : fb ? launch_scan_ffbs(a, *fb, c->stream, &c->launches)
          : launch_scan(a, c->stream, &c->launches));
  if (a.table_upload) c->scan_key.swap(c->scan_key_pending);
  c->scan_key_pending.clear();
  return 0;
}

static KfViews scan_kf_views(const bdlm_problem *p, const bdlm_kf_out *kf) {
  const int64_t n = p->n, R = rows_of(*p);
  KfViews v{};
  if (!kf) return v;
  v.m = mk_view(kf->m, p->layout, 0, 1, R, n); v.C = mk_view(kf->C, p->layout, 0, 1, R, n * n);
  v.a = mk_view(kf->a, p->layout, 0, 1, R, n); v.R = mk_view(kf->R, p->layout, 0, 1, R, n * n);
  v.f = mk_view(kf->f, p->layout, 0, 1, R, 1); v.Q = mk_view(kf->Q, p->layout, 0, 1, R, 1);
  return v;
}

int bdlm_scan_elem_doubles(int32_t n, int32_t backward) {
  if (n < 1 || n > 4) return BDLM_E_ARG;
  return backward ? scan_backward_elem_doubles(n) : scan_forward_elem_doubles(n);
}

int bdlm_scan_combine(int32_t n, int32_t backward, const double *earlier, const double *later,
                      double *out) {
  if (n < 1 || n > 4 || !earlier || !later || !out) return BDLM_E_ARG;
  scan_combine_host(n, backward != 0, earlier, later, out);
  return 0;
}

int bdlm_scan_filter_smooth(bdlm_ctx *c, const bdlm_problem *p, const bdlm_kf_out *kf,
                            const bdlm_smooth_out *sm, int32_t *status) {
  NvtxRange nvtx_("bdlm_scan_filter_smooth");
  int rc = scan_validate(c, p);
  if (rc) return rc;
  if (!sm) return fail(c, BDLM_E_ARG, "null smoother output struct");
  CU(cudaSetDevice(c->device));
  const int64_t n = p->n, R = rows_of(*p);
  bdlm_kf_out k{};
  if (kf) k = *kf;
  // arena: [forward scan workspace | backward scan workspace | (m, C) spill when not wanted]
  const size_t ws = align_up(scan_workspace_bytes(p->n, p->T) + 4096);
  const size_t need = 2 * ws + (k.m ? 0 : align_up(sizeof(double) * R * n)) +
                      (k.C ? 0 : align_up(sizeof(double) * R * n * n)) + 4096;
  rc = ensure_arena(c, need);
  if (rc) return rc;
  Bump bump{c->arena, 2 * ws, c->arena_bytes};
  if (!k.m) k.m = bump.take<double>((size_t)R * n);
  if (!k.C) k.C = bump.take<double>((size_t)R * n * n);
  std::vector<double> prior((size_t)n + n * n);
  std::copy(p->m0, p->m0 + n, prior.begin());
  std::copy(p->C0, p->C0 + n * n, prior.begin() + n);
  ScanArgs a;
  rc = scan_fill(c, p, a, true);
  if (rc) return rc;
  // forward: filter outputs + the smoother's level-1 aggregates (fused into the apply sweep)
  a.phase = kScanApply; a.start = prior.data();
  a.kf = scan_kf_views(p, &k); a.status = status; a.workspace = c->arena;
  a.fuse_sagg = R > 1 ? c->arena + ws : nullptr;
  if (status) CU(cudaMemsetAsync(status, 0, sizeof(int32_t), c->stream));
  { rc = scan_launch_fwd(c, a); if (rc) return rc; }
  // backward: scan the aggregates, apply
  rc = scan_fill(c, p, a);
  if (rc) return rc;
  a.backward = 1; a.phase = kScanApply; a.has_successor = 0;
  a.kf = scan_kf_views(p, &k);
  a.s = mk_view(sm->s, p->layout, 0, 1, R, n); a.S = mk_view(sm->S, p->layout, 0, 1, R, n * n);
  a.status = status; a.workspace = c->arena + ws;
  CU(launch_scan(a, c->stream, &c->launches));
  return 0;
}

int bdlm_scan_loglik(bdlm_ctx *c, const bdlm_problem *p, double *m_last, double *C_last,
                     double *transition, double *innovations, int32_t *status) {
  NvtxRange nvtx_("bdlm_scan_loglik");
  int rc = scan_validate(c, p);
  if (rc) return rc;
  if (p->v_tv || p->w_tv) return fail(c, BDLM_E_ARG, "scan path: time-invariant model (v_tv = w_tv = 0)");
  if (!m_last && !C_last && !transition && !innovations) return fail(c, BDLM_E_ARG, "nothing requested");
  CU(cudaSetDevice(c->device));
  const int64_t n = p->n;
  // arena: [forward scan workspace | block partials + last state]
  const size_t ws = align_up(scan_workspace_bytes(p->n, p->T) + 4096);
  rc = ensure_arena(c, ws + align_up(scan_loglik_bytes(p->n, p->T)) + 4096);
  if (rc) return rc;
  bdlm_problem q = *p;
  q.keep_init = 1;  // as bdlm_loglik: the state (m0, C0) is row 0, every observation a step
  std::vector<double> prior((size_t)n + n * n);
  std::copy(p->m0, p->m0 + n, prior.begin());
  std::copy(p->C0, p->C0 + n * n, prior.begin() + n);
  ScanArgs a;
  rc = scan_fill(c, &q, a, true);
  if (rc) return rc;
  a.phase = kScanApply; a.start = prior.data(); a.workspace = c->arena;
  const ScanLoglikOut o{transition, innovations, m_last, C_last, status, c->arena + ws};
  return scan_launch_fwd(c, a, &o);
}

int bdlm_scan_ffbs(bdlm_ctx *c, const bdlm_problem *p, const double *z, double *theta,
                   const bdlm_kf_out *kf, const bdlm_gibbs_stats *stats, int32_t *status) {
  NvtxRange nvtx_("bdlm_scan_ffbs");
  int rc = scan_validate(c, p);
  if (rc) return rc;
  if (p->v_tv || p->w_tv) return fail(c, BDLM_E_ARG, "scan path: time-invariant model (v_tv = w_tv = 0)");
  if (!p->keep_init) return fail(c, BDLM_E_ARG, "scan FFBS: keep_init = 1");
  if (!theta) return fail(c, BDLM_E_ARG, "null theta");  // z == NULL: on-device Philox normals
  CU(cudaSetDevice(c->device));
  const int64_t n = p->n, R = rows_of(*p);
  bdlm_kf_out k{};
  if (kf) k = *kf;
  // arena: [forward scan workspace | sampler scan workspace | statistics partials | (m, C) spill
  // when not wanted]
  const size_t ws = align_up(scan_workspace_bytes(p->n, p->T) + 4096);
  const size_t parts = align_up(scan_ffbs_parts_bytes(p->n, p->T));
  const size_t need = 2 * ws + parts + (k.m ? 0 : align_up(sizeof(double) * R * n)) +
                      (k.C ? 0 : align_up(sizeof(double) * R * n * n)) + 4096;
  rc = ensure_arena(c, need);
  if (rc) return rc;
  Bump bump{c->arena, 2 * ws + parts, c->arena_bytes};
  if (!k.m) k.m = bump.take<double>((size_t)R * n);
  if (!k.C) k.C = bump.take<double>((size_t)R * n * n);
  std::vector<double> prior((size_t)n + n * n);
  std::copy(p->m0, p->m0 + n, prior.begin());
  std::copy(p->C0, p->C0 + n * n, prior.begin() + n);
  ScanArgs a;
  rc = scan_fill(c, p, a, true);
  if (rc) return rc;
  a.phase = kScanApply; a.start = prior.data(); a.workspace = c->arena;
  a.kf = scan_kf_views(p, &k); a.status = status;
  ScanFfbsOut o{};
  o.z = mk_cview(z, p->layout, 0, 1, R, n);
  o.theta = mk_view(theta, p->layout, 0, 1, R, n);
  if (stats) {
    o.stats.ssy = mk_rowview(stats->ssy, p->layout, 0, 1, 1);
    o.stats.ny = mk_rowview(stats->ny, p->layout, 0, 1, 1);
    o.stats.ssw = mk_rowview(stats->ssw, p->layout, 0, 1, n);
    o.stats.scatter = mk_rowview(stats->scatter, p->layout, 0, 1, n * n);
  }
  o.rng_seed = c->rng_seed; o.rng_sweep = c->rng_sweep; o.rng_base = c->rng_first;
  o.workspace = c->arena + ws;
  o.parts = reinterpret_cast<double *>(c->arena + 2 * ws);
  if (status) CU(cudaMemsetAsync(status, 0, sizeof(int32_t), c->stream));
  return scan_launch_fwd(c, a, nullptr, &o);
}

// ---- device-side multi-GPU protocol for the scan (no host round trip) --------------------
// arena: [forward scan workspace | backward scan workspace]; it must survive from the local to
// the finish phase, so all four calls size it identically.

static int scan_dist_common(bdlm_ctx *c, const bdlm_problem *p, const bdlm_kf_out *kf, int rank,
                            int world, size_t *ws_out) {
  int rc = scan_validate(c, p);
  if (rc) return rc;
  if (world < 1 || rank < 0 || rank >= world) return fail(c, BDLM_E_ARG, "bad rank / world");
  if ((p->keep_init != 0) != (rank == 0))
    return fail(c, BDLM_E_ARG, "time-sharded scan: keep_init = 1 on rank 0 only");
  if (kf && (!kf->m || !kf->C)) return fail(c, BDLM_E_ARG, "time-sharded scan needs kf->m and kf->C");
  CU(cudaSetDevice(c->device));
  const size_t ws = align_up(scan_workspace_bytes(p->n, p->T) + 4096);
  rc = ensure_arena(c, 2 * ws + 4096);
  if (rc) return rc;
  *ws_out = ws;
  return 0;
}

int bdlm_scan_dist_forward_local(bdlm_ctx *c, const bdlm_problem *p, int32_t rank, int32_t world,
                                 double *agg_dev) {
  NvtxRange nvtx_("bdlm_scan_dist_forward_local");
  size_t ws;
  int rc = scan_dist_common(c, p, nullptr, rank, world, &ws);
  if (rc) return rc;
  if (!agg_dev) return fail(c, BDLM_E_ARG, "null aggregate pointer");
  ScanArgs a;
  rc = scan_fill(c, p, a, true);
  if (rc) return rc;
  a.phase = kScanDistLocal; a.agg_dev = agg_dev; a.workspace = c->arena;
  a.rank = rank; a.world = world; a.peers = c->scan_peers; a.epoch_dev = c->scan_epoch;
  { rc = scan_launch_fwd(c, a); if (rc) return rc; }
  return 0;
}

int bdlm_scan_dist_forward_finish(bdlm_ctx *c, const bdlm_problem *p, int32_t rank, int32_t world,
                                  const double *aggs_dev, const bdlm_kf_out *kf, int32_t *status) {
  NvtxRange nvtx_("bdlm_scan_dist_forward_finish");
  size_t ws;
  if (!kf) return fail(c, BDLM_E_ARG, "null output struct");
  int rc = scan_dist_common(c, p, kf, rank, world, &ws);
  if (rc) return rc;
  if (!aggs_dev) return fail(c, BDLM_E_ARG, "null aggregates pointer");
  std::vector<double> prior((size_t)p->n + p->n * p->n);
  std::copy(p->m0, p->m0 + p->n, prior.begin());
  std::copy(p->C0, p->C0 + p->n * p->n, prior.begin() + p->n);
  ScanArgs a;
  rc = scan_fill(c, p, a, true);
  if (rc) return rc;
  a.phase = kScanDistFinish; a.aggs_dev = aggs_dev; a.rank = rank; a.world = world;
  a.peers = c->scan_peers; a.epoch_dev = c->scan_epoch;
  a.start = prior.data(); a.has_successor = rank < world - 1;
  a.kf = scan_kf_views(p, kf); a.status = status; a.workspace = c->arena;
  a.fuse_sagg = c->arena + ws;  // smoother level-1 aggregates for the backward phases
  if (status) CU(cudaMemsetAsync(status, 0, sizeof(int32_t), c->stream));
  { rc = scan_launch_fwd(c, a); if (rc) return rc; }
  return 0;
}

int bdlm_scan_dist_backward_local(bdlm_ctx *c, const bdlm_problem *p, int32_t rank, int32_t world,
                                  const bdlm_kf_out *filt, const bdlm_smooth_out *sm,
                                  double *agg_dev) {
  NvtxRange nvtx_("bdlm_scan_dist_backward_local");
  size_t ws;
  if (!filt) return fail(c, BDLM_E_ARG, "null filtered-state struct");
  int rc = scan_dist_common(c, p, filt, rank, world, &ws);
  if (rc) return rc;
  if (!agg_dev || !sm) return fail(c, BDLM_E_ARG, "null aggregate pointer or output struct");
  const int64_t n = p->n, R = rows_of(*p);
  ScanArgs a;
  rc = scan_fill(c, p, a);
  if (rc) return rc;
  a.backward = 1; a.phase = kScanDistLocal; a.has_successor = rank < world - 1;
  a.kf = scan_kf_views(p, filt);
  a.s = mk_view(sm->s, p->layout, 0, 1, R, n); a.S = mk_view(sm->S, p->layout, 0, 1, R, n * n);
  a.agg_dev = agg_dev; a.rank = rank; a.world = world; a.workspace = c->arena + ws;
  a.peers = c->scan_peers; a.epoch_dev = c->scan_epoch;
  CU(launch_scan(a, c->stream, &c->launches));
  return 0;
}

int bdlm_scan_dist_backward_finish(bdlm_ctx *c, const bdlm_problem *p, int32_t rank, int32_t world,
                                   const double *aggs_dev, const bdlm_kf_out *filt,
                                   const bdlm_smooth_out *sm, int32_t *status) {
  NvtxRange nvtx_("bdlm_scan_dist_backward_finish");
  size_t ws;
  if (!filt) return fail(c, BDLM_E_ARG, "null filtered-state struct");
  int rc = scan_dist_common(c, p, filt, rank, world, &ws);
  if (rc) return rc;
  if (!aggs_dev || !sm) return fail(c, BDLM_E_ARG, "null aggregates pointer or output struct");
  const int64_t n = p->n, R = rows_of(*p);
  ScanArgs a;
  rc = scan_fill(c, p, a);
  if (rc) return rc;
  a.backward = 1; a.phase = kScanDistFinish; a.has_successor = rank < world - 1;
  a.kf = scan_kf_views(p, filt);
  a.s = mk_view(sm->s, p->layout, 0, 1, R, n); a.S = mk_view(sm->S, p->layout, 0, 1, R, n * n);
  a.aggs_dev = aggs_dev; a.rank = rank; a.world = world; a.status = status;
  a.workspace = c->arena + ws; a.peers = c->scan_peers; a.epoch_dev = c->scan_epoch;
  CU(launch_scan(a, c->stream, &c->launches));
  return 0;
}

// ---- "next" rows: scalar AR(1) / OU, conjugate filter, conjugate draws -------------------

static int ar_call(bdlm_ctx *c, int op, const bdlm_ar_problem *ap, const bdlm_ar_out *out,
                   const double *z, double *theta) {
  static const double one = 1.0;
  if (!c) return fail(nullptr, BDLM_E_ARG, "null context");
  if (!ap) return fail(c, BDLM_E_ARG, "null problem");
  if (ap->T == 0) return fail(c, BDLM_E_EMPTY, "T == 0: empty observation vector");
  if (ap->process != BDLM_AR1 && ap->process != BDLM_OU) return fail(c, BDLM_E_ARG, "bad process");
  if (ap->v_mode < BDLM_V_SCALAR || ap->v_mode > BDLM_V_PER_SERIES_STEP)
    return fail(c, BDLM_E_ARG, "bad v_mode");
  if (!ap->phi || !ap->mu || !ap->sigma_eta || !ap->v || !ap->y)
    return fail(c, BDLM_E_ARG, "null phi, mu, sigma_eta, v or y");
  if (op == A_AR_FFBS && (!z || !theta)) return fail(c, BDLM_E_ARG, "null z or theta");
  if (op == A_AR_FILTER && !out) return fail(c, BDLM_E_ARG, "null output struct");
  DevCall d{};
  d.op = op;
  d.pr.B = ap->B; d.pr.T = ap->T; d.pr.n = 1; d.pr.p = 1; d.pr.layout = ap->layout;
  d.pr.mem = ap->mem; d.pr.keep_init = 1; d.pr.times = ap->times; d.pr.y = ap->y;
  d.pr.F = d.pr.G = d.pr.V = d.pr.W = d.pr.m0 = d.pr.C0 = &one;
  int rc = validate(c, A_FILTER, &d.pr);
  if (rc) return rc;
  d.ar = *ap;
  if (out) d.ar_out = *out;
  d.z = z; d.theta = theta;
  return dispatch(c, d);
}

int bdlm_ar_filter(bdlm_ctx *c, const bdlm_ar_problem *ap, const bdlm_ar_out *out) {
  NvtxRange nvtx_("bdlm_ar_filter");
  return ar_call(c, A_AR_FILTER, ap, out, nullptr, nullptr);
}

int bdlm_ar_ffbs(bdlm_ctx *c, const bdlm_ar_problem *ap, const double *z, double *theta,
                 const bdlm_ar_out *filt) {
  NvtxRange nvtx_("bdlm_ar_ffbs");
  return ar_call(c, A_AR_FFBS, ap, filt, z, theta);
}

int bdlm_conjugate_filter(bdlm_ctx *c, const bdlm_problem *p, double prior_shape,
                          double prior_scale, const bdlm_kf_out *out, double *shape,
                          double *scale, int32_t *status) {
  NvtxRange nvtx_("bdlm_conjugate_filter");
  int rc = validate(c, A_CONJ_FILTER, p);
  if (rc) return rc;
  if (!conjugate_supported(p->n, p->p) || p->f_tv || p->g_tv || !p->keep_init)
    return fail(c, BDLM_E_ARG,
                "conjugate filter: p = 1, n <= 4, time-invariant F and G, keep_init = 1");
  DevCall d{}; d.op = A_CONJ_FILTER; d.pr = *p;
  d.pr.per_series &= ~BDLM_PS_V;  // V is what the filter learns
  d.pr.V = nullptr;
  if (out) d.kf = *out;
  d.cj_shape = prior_shape; d.cj_scale = prior_scale;
  d.cj_shape_out = shape; d.cj_scale_out = scale;
  d.status = status;
  return dispatch(c, d);
}

int bdlm_gibbs_draw(bdlm_ctx *c, const bdlm_problem *p, const bdlm_gibbs_stats *stats,
                    const bdlm_gibbs_prior *prior, const bdlm_gibbs_rng *rng, double *V_out,
                    double *W_out, double *v_shape_rate, double *w_shape_rate, int32_t *status) {
  NvtxRange nvtx_("bdlm_gibbs_draw");
  int rc = validate(c, A_GIBBS_DRAW, p);
  if (rc) return rc;
  if (!stats || !prior || !rng) return fail(c, BDLM_E_ARG, "null stats, prior or rng");
  if (V_out && (!stats->ssy || !stats->ny)) return fail(c, BDLM_E_ARG, "V draw needs ssy and ny");
  if (W_out && !prior->w_psi && !stats->ssw) return fail(c, BDLM_E_ARG, "diagonal W draw needs ssw");
  if (W_out && prior->w_psi && !stats->scatter)
    return fail(c, BDLM_E_ARG, "inverse-Wishart W draw needs the scatter matrix");
  if (!W_out && prior->w_psi) return fail(c, BDLM_E_ARG, "inverse-Wishart prior without W_out");
  DevCall d{}; d.op = A_GIBBS_DRAW; d.pr = *p;
  d.stats = *stats; d.prior = *prior; d.rng = *rng;
  d.V_out = V_out; d.W_out = W_out; d.v_sr = v_shape_rate; d.w_sr = w_shape_rate;
  d.status = status;
  return dispatch(c, d);
}

int bdlm_gibbs_suffstats(bdlm_ctx *c, const bdlm_problem *p, const double *theta,
                         const bdlm_gibbs_stats *stats) {
  NvtxRange nvtx_("bdlm_gibbs_suffstats");
  int rc = validate(c, A_STATS, p);
  if (rc) return rc;
  if (!theta || !stats) return fail(c, BDLM_E_ARG, "null theta or stats");
  DevCall d{}; d.op = A_STATS; d.pr = *p; d.theta = const_cast<double *>(theta);
  d.stats = *stats;
  return dispatch(c, d);
}

}  // extern "C"
