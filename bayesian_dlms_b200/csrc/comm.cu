// comm.cu -- multi-GPU communicator of libbdlm.so (include/bdlm.h, "multi-GPU" section).
//
// SURVEY.md 8(b) "Threading": one context per device; a communicator object wraps NCCL init and the
// per-device contexts.  Series and chains are independent (the reference's own multi-series
// workflow fits one model per sensor, UoModel.scala:69-104; its only parallel driver maps chains
// over futures, Streaming.scala:162-173), so the data path has NO collective: a batch is cut into
// contiguous blocks of series, one per device.  The only inter-GPU traffic is
//   * an ncclAllReduce of sums of log-likelihoods / pooled Gibbs sufficient statistics, and
//   * for ONE long series cut along time (BASELINE config 5), the chunk aggregates of the
//     associative scan: 3n^2+2n doubles per rank forwards, 2n^2+n backwards.  They travel either
//     through NCCL all-gathers or -- when every peer's mailbox is mapped into this process
//     (single-process communicators with peer access) -- by direct NVLink stores from the kernel
//     that produced them, with a release flag the consuming kernel spins on (scan.cu).
//
// Two ways to build a communicator with the same entry point (bdlm_comm_create):
//   * single process, n devices (a JVM host driving all GPUs of a node): id == NULL,
//     n_local == world -> ncclCommInitAll; sharded calls run one host thread per device;
//   * one process per GPU (torchrun / MPI style): every process passes the 128-byte id rank 0 got
//     from bdlm_comm_unique_id -> ncclCommInitRank.
//
// NCCL is loaded at run time (dlopen "libnccl.so.2"): libbdlm.so has no link-time dependency on it,
// and inside a PyTorch process the copy torch already loaded is the one that is used.
#include <dlfcn.h>

#include <algorithm>
#include <condition_variable>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "common.cuh"
#include "ctx_internal.h"
#include "launch.h"

using namespace bdlm;

namespace {

// ---- the few NCCL entry points used, resolved with dlsym (ABI-stable across NCCL 2.x) -------
typedef struct ncclComm *nccl_comm_t;
struct nccl_uid { char internal[128]; };
enum { kNcclSum = 0, kNcclInt8 = 0, kNcclFloat64 = 8 };

struct Nccl {
  void *h = nullptr;
  int (*GetUniqueId)(nccl_uid *) = nullptr;
  int (*CommInitRank)(nccl_comm_t *, int, nccl_uid, int) = nullptr;
  int (*CommInitAll)(nccl_comm_t *, int, const int *) = nullptr;
  int (*CommDestroy)(nccl_comm_t) = nullptr;
  int (*AllReduce)(const void *, void *, size_t, int, int, nccl_comm_t, cudaStream_t) = nullptr;
  int (*AllGather)(const void *, void *, size_t, int, nccl_comm_t, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char *(*GetErrorString)(int) = nullptr;
  std::string err;
};

void nccl_load(Nccl &g) {
  const char *names[] = {std::getenv("BDLM_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
  std::string why;
  for (const char *nm : names) {
    if (!nm || !*nm) continue;
    g.h = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
    if (g.h) break;
    const char *e = dlerror();  // one call: dlerror() clears the message it returns
    if (e) why = e;
  }
  if (!g.h) { g.err = "cannot load NCCL (libnccl.so.2): " + why; return; }
#define SYM(field, name)                                                       \
  *reinterpret_cast<void **>(&g.field) = dlsym(g.h, name);                     \
  if (!g.field) { g.err = std::string("NCCL symbol missing: ") + name; g.h = nullptr; return; }
  SYM(GetUniqueId, "ncclGetUniqueId") SYM(CommInitRank, "ncclCommInitRank")
  SYM(CommInitAll, "ncclCommInitAll") SYM(CommDestroy, "ncclCommDestroy")
  SYM(AllReduce, "ncclAllReduce") SYM(AllGather, "ncclAllGather")
  SYM(GroupStart, "ncclGroupStart") SYM(GroupEnd, "ncclGroupEnd")
  SYM(GetErrorString, "ncclGetErrorString")
#undef SYM
}

Nccl *nccl() {
  // function-local static: initialised once, thread-safe (communicators may be created from
  // several host threads)
  static Nccl *g = [] { Nccl *x = new Nccl(); nccl_load(*x); return x; }();
  return g;
}

constexpr int kMaxElem = 3 * 4 * 4 + 2 * 4;  // forward scan element at n = 4 (56 doubles)
constexpr int kRedMax = 4096;                // doubles per all-reduce through the device buffer

struct Local {
  int device = 0, rank = 0;
  bdlm_ctx *ctx = nullptr;
  nccl_comm_t nc = nullptr;
  double *red = nullptr;     // device [kRedMax]: all-reduce staging
  double *agg = nullptr;     // device [2][kMaxElem]: this rank's scan aggregates (fwd, bwd)
  double *aggs = nullptr;    // device [2][world][kMaxElem]: gathered aggregates / peer mailbox
  unsigned long long *flags = nullptr;  // device [2][world] mailbox flags, then [1]: this rank's call counter
  // device [kXch][kMaxElem] send slots, then [kXch][world][kMaxElem] gathered: the NCCL exchanges of
  // the time-sharded log-likelihoods and FFBS.  Not agg / aggs: on a mailbox communicator those are
  // the peers' store targets, and a peer that already runs the next filter + smoother could publish
  // into a slot this rank's all-gather is still writing.
  double *xch = nullptr;
};
constexpr int kXch = 3;  // exchanges of one call at most (FFBS: forward aggregates, sampler aggregates, partials)

// One persistent host thread per local device: a single thread enqueuing ~20 launches per device
// is the bottleneck of a multi-GPU call (measured at 8 GPUs: 0.64 ms of host enqueue for 0.2 ms of
// kernels per device), and creating threads per call would cost as much again.
struct Worker {
  std::thread th;
  std::mutex mu;
  std::condition_variable cv;
  std::function<int()> job;
  int rc = 0;
  bool pending = false, quit = false;
  Worker() { th = std::thread([this] { loop(); }); }
  ~Worker() {
    { std::lock_guard<std::mutex> lk(mu); quit = true; }
    cv.notify_all();
    if (th.joinable()) th.join();
  }
  void loop() {
    std::unique_lock<std::mutex> lk(mu);
    for (;;) {
      cv.wait(lk, [&] { return pending || quit; });
      if (quit) return;
      std::function<int()> j = job;
      lk.unlock();
      const int r = j();
      lk.lock();
      rc = r; pending = false;
      cv.notify_all();
    }
  }
  void submit(std::function<int()> j) {
    { std::lock_guard<std::mutex> lk(mu); job = std::move(j); pending = true; }
    cv.notify_all();
  }
  int wait() {
    std::unique_lock<std::mutex> lk(mu);
    cv.wait(lk, [&] { return !pending; });
    return rc;
  }
};

}  // namespace

struct bdlm_comm {
  int world = 0;
  std::vector<Local> loc;
  std::vector<std::unique_ptr<Worker>> workers;  // one per local device when there are several
  std::string err;
  bool peer = false;               // every local device can store into every other's mailbox
  ScanPeers peers[2]{};            // [forward, backward] mailbox tables for scan.cu
};

static std::string g_comm_err;

namespace {

int cfail(bdlm_comm *m, int code, const std::string &msg) {
  if (m) m->err = msg; else g_comm_err = msg;
  return code;
}

#define CCU(call)                                                                          \
  do {                                                                                     \
    cudaError_t e_ = (call);                                                               \
    if (e_ != cudaSuccess)                                                                 \
      return cfail(m, BDLM_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));    \
  } while (0)
#define CNC(call)                                                                          \
  do {                                                                                     \
    int r_ = (call);                                                                       \
    if (r_ != 0)                                                                           \
      return cfail(m, BDLM_E_NCCL, std::string(#call) + ": " + nccl()->GetErrorString(r_)); \
  } while (0)

// sum of x[lo..hi) per component k of a one-row-per-series array ([k][B] or [B][k]) on the host
void host_partial(const double *x, int layout, int64_t B, int64_t lo, int64_t hi, int k, double *out) {
  for (int c = 0; c < k; ++c) {
    double acc = 0.0;
    if (layout == BDLM_TIME_MAJOR) { const double *p = x + (int64_t)c * B; for (int64_t b = lo; b < hi; ++b) acc += p[b]; }
    else for (int64_t b = lo; b < hi; ++b) acc += x[b * k + c];
    out[c] = acc;
  }
}

// one block per component: deterministic strided partial sums + shared-memory tree
__global__ void __launch_bounds__(256)
colsum_kernel(const double *__restrict__ x, int64_t sb, int64_t sk, int64_t lo, int64_t hi,
              double *__restrict__ out) {
  __shared__ double sh[256];
  const double *p = x + (int64_t)blockIdx.x * sk;
  double acc = 0.0;
  for (int64_t b = lo + threadIdx.x; b < hi; b += 256) acc += p[b * sb];
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[blockIdx.x] = sh[0];
}

// Partial sums of this process's series into Local.red[off..off+k) of every local device, for a
// one-row-per-series array x (NULL = zeros).  Host arrays: summed on the host and uploaded; device
// arrays (n_local == 1): reduced by a kernel on the context's stream.
int stage_partial(bdlm_comm *m, const double *x, const bdlm_problem *p, int k, int off,
                  const std::vector<int64_t> &cut) {
  for (size_t i = 0; i < m->loc.size(); ++i) {
    Local &L = m->loc[i];
    CCU(cudaSetDevice(L.device));
    cudaStream_t st = ctx_stream(L.ctx);
    if (!x) { CCU(cudaMemsetAsync(L.red + off, 0, sizeof(double) * k, st)); continue; }
    if (p->mem == BDLM_HOST) {
      std::vector<double> part(k);
      host_partial(x, p->layout, p->B, cut[i], cut[i + 1], k, part.data());
      CCU(cudaMemcpyAsync(L.red + off, part.data(), sizeof(double) * k, cudaMemcpyHostToDevice, st));
      CCU(cudaStreamSynchronize(st));  // `part` is pageable and about to go out of scope
    } else {
      const int64_t sb = p->layout == BDLM_TIME_MAJOR ? 1 : k, sk = p->layout == BDLM_TIME_MAJOR ? p->B : 1;
      colsum_kernel<<<k, 256, 0, st>>>(x, sb, sk, cut[i], cut[i + 1], L.red + off);
      CCU(cudaGetLastError());
      ctx_count_launches(L.ctx, 1);
    }
  }
  return 0;
}

// ncclAllReduce(sum) of red[0..count) over ALL ranks, then device rank-local-0 -> host out
int allreduce_staged(bdlm_comm *m, int count, double *out) {
  Nccl *nc = nccl();
  CNC(nc->GroupStart());
  for (Local &L : m->loc) {
    int r = nc->AllReduce(L.red, L.red, (size_t)count, kNcclFloat64, kNcclSum, L.nc, ctx_stream(L.ctx));
    if (r != 0) { nc->GroupEnd(); return cfail(m, BDLM_E_NCCL, std::string("ncclAllReduce: ") + nc->GetErrorString(r)); }
  }
  CNC(nc->GroupEnd());
  Local &L0 = m->loc[0];
  CCU(cudaSetDevice(L0.device));
  CCU(cudaMemcpyAsync(out, L0.red, sizeof(double) * count, cudaMemcpyDeviceToHost, ctx_stream(L0.ctx)));
  for (Local &L : m->loc) {
    CCU(cudaSetDevice(L.device));
    CCU(cudaStreamSynchronize(ctx_stream(L.ctx)));
  }
  return 0;
}

// contiguous blocks of this process's series, one per local device
std::vector<int64_t> cuts(const bdlm_comm *m, int64_t B) {
  const int n = (int)m->loc.size();
  std::vector<int64_t> c(n + 1);
  for (int i = 0; i <= n; ++i) c[i] = B * i / n;
  return c;
}

// Run fn(local index) for every local device: directly when there is one, else one host thread each
// (the slab pipeline of a host-buffer call blocks its thread while copies and kernels overlap).
template <class Fn>
int for_each_local(bdlm_comm *m, Fn fn) {
  const int n = (int)m->loc.size();
  std::vector<int> rc(n, 0);
  if (n == 1) rc[0] = fn(0);
  else {
    for (int i = 0; i < n; ++i) m->workers[i]->submit([&fn, i] { return fn(i); });
    for (int i = 0; i < n; ++i) rc[i] = m->workers[i]->wait();
  }
  int worst = 0, numeric = 0;
  for (int i = 0; i < n; ++i) {
    if (rc[i] < 0 && worst == 0) {
      worst = rc[i];
      m->err = std::string("device ") + std::to_string(m->loc[i].device) + ": " + bdlm_last_error(m->loc[i].ctx);
    }
    if (rc[i] > 0) numeric += rc[i];
  }
  return worst ? worst : numeric;
}

// The sub-batch [lo, hi) of the NEXT call on a context.  dispatch() consumes it, but a call that
// fails validation never gets there: the guard clears it on every path, so a later direct call on
// the same context (bdlm_comm_ctx) cannot inherit a stale shard.
struct ShardRange {
  bdlm_ctx *c;
  ShardRange(bdlm_ctx *ctx, int64_t lo, int64_t hi) : c(ctx) { ctx_set_range(c, lo, hi); }
  ~ShardRange() { ctx_set_range(c, -1, -1); }
  ShardRange(const ShardRange &) = delete;
  ShardRange &operator=(const ShardRange &) = delete;
};

int check_sharded(bdlm_comm *m, const bdlm_problem *p) {
  if (!m) return cfail(nullptr, BDLM_E_ARG, "null communicator");
  if (!p) return cfail(m, BDLM_E_ARG, "null problem");
  if (p->mem == BDLM_DEVICE && m->loc.size() != 1)
    return cfail(m, BDLM_E_ARG, "device-resident batches need one device per process: pass host "
                                "buffers to a single-process communicator");
  return 0;
}

// ---- helpers of the time-sharded log-likelihoods and FFBS (bdlm_comm_scan_loglik / _ffbs)

// Checks every local chunk before any device work: a rank that failed after its peers had entered
// an all-gather would leave them waiting.
int check_scan_chunks(bdlm_comm *m, const bdlm_problem *probs, const int64_t *first_row, int64_t total_T) {
  if (!m) return cfail(nullptr, BDLM_E_ARG, "null communicator");
  if (!probs) return cfail(m, BDLM_E_ARG, "null problem array");
  const int n = probs[0].n;
  if (n < 1 || n > 4) return cfail(m, BDLM_E_ARG, "scan path: n <= 4");
  for (size_t i = 0; i < m->loc.size(); ++i) {
    const bdlm_problem &p = probs[i];
    const int rank = m->loc[i].rank;
    if (p.n != n) return cfail(m, BDLM_E_ARG, "time-sharded scan: every chunk describes the same model (n differs)");
    if ((p.keep_init != 0) != (rank == 0)) return cfail(m, BDLM_E_ARG, "time-sharded scan: keep_init = 1 on rank 0 only");
    if (p.T < 1) return cfail(m, BDLM_E_ARG, "time-sharded scan: every chunk holds at least one observation");
    if (first_row && ((first_row[i] == 0) != (rank == 0) || first_row[i] < 0 ||
                      first_row[i] + p.T + p.keep_init > total_T + 1))
      return cfail(m, BDLM_E_ARG, "time-sharded FFBS: first_row = 0 on rank 0 only, first_row + rows <= total_T + 1");
  }
  return 0;
}

double *xch_send(const Local &L, int k) { return L.xch + (size_t)k * kMaxElem; }
double *xch_recv(const Local &L, int world, int k) { return L.xch + (size_t)kXch * kMaxElem + (size_t)k * world * kMaxElem; }

template <class P>
P entry(P const *arr, int i) { return arr ? arr[i] : nullptr; }

// ncclAllGather of `count` doubles from send slot k into the gathered slot k, on the context's stream
int xch_gather(const Local &L, int world, int k, int count) {
  return nccl()->AllGather(xch_send(L, k), xch_recv(L, world, k), (size_t)count, kNcclFloat64, L.nc,
                           ctx_stream(L.ctx)) == 0 ? 0 : BDLM_E_NCCL;
}

}  // namespace

extern "C" {

int bdlm_comm_unique_id(void *id) {
  bdlm_comm *m = nullptr;
  if (!id) return cfail(nullptr, BDLM_E_ARG, "null id");
  Nccl *nc = nccl();
  if (!nc->h) return cfail(nullptr, BDLM_E_NCCL, nc->err);
  nccl_uid u;
  CNC(nc->GetUniqueId(&u));
  std::memcpy(id, u.internal, BDLM_COMM_ID_BYTES);
  return 0;
}

void bdlm_comm_destroy(bdlm_comm *m) {
  if (!m) return;
  m->workers.clear();  // joins the worker threads
  for (Local &L : m->loc) {
    cudaSetDevice(L.device);
    if (L.ctx) bdlm_sync(L.ctx);
    if (L.nc) nccl()->CommDestroy(L.nc);
    if (L.red) cudaFree(L.red);
    if (L.agg) cudaFree(L.agg);
    if (L.aggs) cudaFree(L.aggs);
    if (L.flags) cudaFree(L.flags);
    if (L.xch) cudaFree(L.xch);
    if (L.ctx) bdlm_destroy(L.ctx);
  }
  delete m;
}

int bdlm_comm_create(const int32_t *devices, int32_t n_local, int32_t first_rank, int32_t world,
                     const void *id, bdlm_comm **out) {
  bdlm_comm *m = nullptr;
  if (!out) return cfail(nullptr, BDLM_E_ARG, "null out pointer");
  *out = nullptr;
  if (!devices || n_local < 1 || world < n_local || first_rank < 0 || first_rank + n_local > world)
    return cfail(nullptr, BDLM_E_ARG, "bad device list / rank range");
  if (!id && n_local != world)
    return cfail(nullptr, BDLM_E_ARG, "a communicator spanning several processes needs the id "
                                      "from bdlm_comm_unique_id");
  if (world > BDLM_COMM_MAX_WORLD) return cfail(nullptr, BDLM_E_ARG, "world size above BDLM_COMM_MAX_WORLD");
  Nccl *nc = nccl();
  if (!nc->h) return cfail(nullptr, BDLM_E_NCCL, nc->err);
  m = new (std::nothrow) bdlm_comm();
  if (!m) return cfail(nullptr, BDLM_E_ARG, "out of host memory");
  m->world = world;
  m->loc.resize(n_local);
  auto bail = [&](int code, const std::string &msg) {
    g_comm_err = msg;
    bdlm_comm_destroy(m);
    return code;
  };
  for (int i = 0; i < n_local; ++i) {
    Local &L = m->loc[i];
    L.device = devices[i]; L.rank = first_rank + i;
    int rc = bdlm_create(L.device, &L.ctx);
    if (rc) return bail(rc, std::string("bdlm_create: ") + bdlm_last_error(nullptr));
    cudaError_t e = cudaSetDevice(L.device);
    if (e == cudaSuccess) e = cudaMalloc(&L.red, sizeof(double) * kRedMax);
    if (e == cudaSuccess) e = cudaMalloc(&L.agg, sizeof(double) * 2 * kMaxElem);
    if (e == cudaSuccess) e = cudaMalloc(&L.aggs, sizeof(double) * 2 * world * kMaxElem);
    if (e == cudaSuccess) e = cudaMalloc(&L.flags, sizeof(unsigned long long) * (2 * world + 1));
    if (e == cudaSuccess) e = cudaMemset(L.flags, 0, sizeof(unsigned long long) * (2 * world + 1));
    if (e == cudaSuccess) e = cudaMalloc(&L.xch, sizeof(double) * kXch * (world + 1) * kMaxElem);
    if (e != cudaSuccess) return bail(BDLM_E_CUDA, std::string("communicator buffers: ") + cudaGetErrorString(e));
  }
  if (!id) {
    std::vector<nccl_comm_t> comms(n_local);
    std::vector<int> devs(devices, devices + n_local);
    int r = nc->CommInitAll(comms.data(), n_local, devs.data());
    if (r != 0) return bail(BDLM_E_NCCL, std::string("ncclCommInitAll: ") + nc->GetErrorString(r));
    for (int i = 0; i < n_local; ++i) m->loc[i].nc = comms[i];
  } else {
    nccl_uid u;
    std::memcpy(u.internal, id, BDLM_COMM_ID_BYTES);
    int r = nc->GroupStart();
    for (int i = 0; i < n_local && r == 0; ++i) {
      cudaSetDevice(m->loc[i].device);
      r = nc->CommInitRank(&m->loc[i].nc, world, u, m->loc[i].rank);
    }
    int r2 = nc->GroupEnd();
    if (r == 0) r = r2;
    if (r != 0) return bail(BDLM_E_NCCL, std::string("ncclCommInitRank: ") + nc->GetErrorString(r));
  }
  // Peer mailboxes for the scan exchange: only when this process drives every rank and each
  // device can address every other one (NVLink / NVSwitch); otherwise NCCL all-gathers are used.
  m->peer = n_local == world && world > 1 && std::getenv("BDLM_COMM_NO_PEER") == nullptr;
  for (int i = 0; i < n_local && m->peer; ++i)
    for (int j = 0; j < n_local && m->peer; ++j) {
      if (i == j) continue;
      int can = 0;
      if (cudaDeviceCanAccessPeer(&can, m->loc[i].device, m->loc[j].device) != cudaSuccess || !can) m->peer = false;
    }
  if (m->peer) {
    for (int i = 0; i < n_local; ++i) {
      cudaSetDevice(m->loc[i].device);
      for (int j = 0; j < n_local; ++j) {
        if (i == j) continue;
        cudaError_t e = cudaDeviceEnablePeerAccess(m->loc[j].device, 0);
        if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); e = cudaSuccess; }
        if (e != cudaSuccess) { cudaGetLastError(); m->peer = false; }
      }
    }
  }
  for (int pass = 0; pass < 2; ++pass) {
    m->peers[pass].world = m->peer ? world : 0;
    for (int r = 0; r < world && m->peer; ++r) {
      m->peers[pass].box[r] = m->loc[r].aggs + (size_t)pass * world * kMaxElem;
      m->peers[pass].flag[r] = m->loc[r].flags + (size_t)pass * world;
    }
  }
  if (n_local > 1)
    for (int i = 0; i < n_local; ++i) m->workers.emplace_back(new Worker());
  *out = m;
  return 0;
}

const char *bdlm_comm_last_error(bdlm_comm *m) { return m ? m->err.c_str() : g_comm_err.c_str(); }
int32_t bdlm_comm_size(bdlm_comm *m) { return m ? m->world : 0; }
int32_t bdlm_comm_local_size(bdlm_comm *m) { return m ? (int32_t)m->loc.size() : 0; }
int32_t bdlm_comm_uses_peer_exchange(bdlm_comm *m) { return m && m->peer ? 1 : 0; }
bdlm_ctx *bdlm_comm_ctx(bdlm_comm *m, int32_t i) {
  return (m && i >= 0 && i < (int32_t)m->loc.size()) ? m->loc[i].ctx : nullptr;
}

int bdlm_comm_allreduce_sum(bdlm_comm *m, double *values, int32_t count) {
  if (!m) return cfail(nullptr, BDLM_E_ARG, "null communicator");
  if (!values || count < 1 || count > kRedMax) return cfail(m, BDLM_E_ARG, "bad values / count");
  // this PROCESS contributes `values` once (through its first device); its other devices add zeros
  for (size_t i = 0; i < m->loc.size(); ++i) {
    Local &L = m->loc[i];
    CCU(cudaSetDevice(L.device));
    if (i == 0) {
      CCU(cudaMemcpyAsync(L.red, values, sizeof(double) * count, cudaMemcpyHostToDevice, ctx_stream(L.ctx)));
      CCU(cudaStreamSynchronize(ctx_stream(L.ctx)));
    } else {
      CCU(cudaMemsetAsync(L.red, 0, sizeof(double) * count, ctx_stream(L.ctx)));
    }
  }
  return allreduce_staged(m, count, values);
}

int bdlm_comm_allreduce_sum_device(bdlm_comm *m, double *values_dev, int32_t count) {
  if (!m) return cfail(nullptr, BDLM_E_ARG, "null communicator");
  if (m->loc.size() != 1) return cfail(m, BDLM_E_ARG, "device all-reduce: one device per process");
  if (!values_dev || count < 1) return cfail(m, BDLM_E_ARG, "bad values / count");
  Local &L = m->loc[0];
  CCU(cudaSetDevice(L.device));
  CNC(nccl()->AllReduce(values_dev, values_dev, (size_t)count, kNcclFloat64, kNcclSum, L.nc, ctx_stream(L.ctx)));
  return 0;  // enqueued on the context's stream, like every device-mode call
}

int bdlm_comm_kf_filter_smooth(bdlm_comm *m, const bdlm_problem *p, const bdlm_kf_out *kf,
                               const bdlm_smooth_out *sm, int32_t *status) {
  int rc = check_sharded(m, p);
  if (rc) return rc;
  const std::vector<int64_t> cut = cuts(m, p->B);
  return for_each_local(m, [&](int i) {
    ShardRange shard_(m->loc[i].ctx, cut[i], cut[i + 1]);
    return bdlm_kf_filter_smooth(m->loc[i].ctx, p, kf, sm, status);
  });
}

int bdlm_comm_kf_filter(bdlm_comm *m, const bdlm_problem *p, const bdlm_kf_out *out, int32_t *status) {
  int rc = check_sharded(m, p);
  if (rc) return rc;
  const std::vector<int64_t> cut = cuts(m, p->B);
  return for_each_local(m, [&](int i) {
    ShardRange shard_(m->loc[i].ctx, cut[i], cut[i + 1]);
    return bdlm_kf_filter(m->loc[i].ctx, p, out, status);
  });
}

int bdlm_comm_svd_filter(bdlm_comm *m, const bdlm_problem *p, const bdlm_svd_out *out, int32_t *status) {
  int rc = check_sharded(m, p);
  if (rc) return rc;
  const std::vector<int64_t> cut = cuts(m, p->B);
  return for_each_local(m, [&](int i) {
    ShardRange shard_(m->loc[i].ctx, cut[i], cut[i + 1]);
    return bdlm_svd_filter(m->loc[i].ctx, p, out, status);
  });
}

int bdlm_comm_loglik(bdlm_comm *m, const bdlm_problem *p, double *transition, double *innovations,
                     int32_t *status, double *sums) {
  int rc = check_sharded(m, p);
  if (rc) return rc;
  const std::vector<int64_t> cut = cuts(m, p->B);
  rc = for_each_local(m, [&](int i) {
    ShardRange shard_(m->loc[i].ctx, cut[i], cut[i + 1]);
    return bdlm_loglik(m->loc[i].ctx, p, transition, innovations, status);
  });
  if (rc < 0 || !sums) return rc;
  // the one collective of this path: Sum_b log-likelihood over every series of every rank
  bdlm_problem row = *p;  // [B] arrays: one component per series
  row.layout = BDLM_SERIES_MAJOR;
  int r2 = stage_partial(m, transition, &row, 1, 0, cut);
  if (!r2) r2 = stage_partial(m, innovations, &row, 1, 1, cut);
  if (!r2) r2 = allreduce_staged(m, 2, sums);
  return r2 ? r2 : rc;
}

static int comm_ffbs(bdlm_comm *m, bool svd, const bdlm_problem *p, const double *z, double *theta,
                     const bdlm_kf_out *kf, const bdlm_svd_out *filt, const bdlm_gibbs_stats *stats,
                     int32_t *status, const bdlm_gibbs_stats *pooled) {
  int rc = check_sharded(m, p);
  if (rc) return rc;
  if (pooled && !stats) return cfail(m, BDLM_E_ARG, "pooled statistics need the per-chain stats arrays");
  const int n = p->n, pp = p->p;
  if (pooled && 2 * pp + n + n * n > kRedMax) return cfail(m, BDLM_E_ARG, "statistics too large");
  if (pooled && ((pooled->ssy && !stats->ssy) || (pooled->ny && !stats->ny) ||
                 (pooled->ssw && !stats->ssw) || (pooled->scatter && !stats->scatter)))
    return cfail(m, BDLM_E_ARG, "pooled statistic requested without its per-chain array");
  const std::vector<int64_t> cut = cuts(m, p->B);
  // chains keep their GLOBAL Philox subsequence whatever the cut (ctx rng_first + index in the call)
  rc = for_each_local(m, [&](int i) {
    ShardRange shard_(m->loc[i].ctx, cut[i], cut[i + 1]);
    return svd ? bdlm_svd_ffbs(m->loc[i].ctx, p, z, theta, filt, stats, status)
               : bdlm_ffbs(m->loc[i].ctx, p, z, theta, kf, stats, status);
  });
  if (rc < 0 || !pooled) return rc;
  // Sum over ALL chains of all ranks of the Gibbs sufficient statistics (Gibbs.scala:29-43,63-73;
  // GibbsWishart.scala:22-29): what a sampler that pools V / W across series conditions on.
  int off = 0, r2 = 0;
  const int sizes[4] = {pp, pp, n, n * n};
  const double *src[4] = {stats->ssy, stats->ny, stats->ssw, stats->scatter};
  double *dst[4] = {pooled->ssy, pooled->ny, pooled->ssw, pooled->scatter};
  for (int f = 0; f < 4 && !r2; ++f) { r2 = stage_partial(m, dst[f] ? src[f] : nullptr, p, sizes[f], off, cut); off += sizes[f]; }
  std::vector<double> tot(off);
  if (!r2) r2 = allreduce_staged(m, off, tot.data());
  if (r2) return r2;
  off = 0;
  for (int f = 0; f < 4; ++f) {
    if (dst[f]) std::memcpy(dst[f], tot.data() + off, sizeof(double) * sizes[f]);
    off += sizes[f];
  }
  return rc;
}

int bdlm_comm_ffbs(bdlm_comm *m, const bdlm_problem *p, const double *z, double *theta,
                   const bdlm_kf_out *kf, const bdlm_gibbs_stats *stats, int32_t *status,
                   const bdlm_gibbs_stats *pooled) {
  return comm_ffbs(m, false, p, z, theta, kf, nullptr, stats, status, pooled);
}

int bdlm_comm_svd_ffbs(bdlm_comm *m, const bdlm_problem *p, const double *z, double *theta,
                       const bdlm_svd_out *filt, const bdlm_gibbs_stats *stats, int32_t *status,
                       const bdlm_gibbs_stats *pooled) {
  return comm_ffbs(m, true, p, z, theta, nullptr, filt, stats, status, pooled);
}

// ---- ONE long series cut along time over the ranks (BASELINE config 5) ---------------------
// probs / kfs / sms / status: one entry per LOCAL device, describing that rank's time chunk in
// its own device memory (keep_init = 1 on global rank 0 only).  Enqueue-only: every phase runs on
// the contexts' streams; call bdlm_sync on the contexts (or bdlm_comm_sync) before reading.
int bdlm_comm_scan_filter_smooth(bdlm_comm *m, const bdlm_problem *probs, const bdlm_kf_out *kfs,
                                 const bdlm_smooth_out *sms, int32_t *const *status) {
  int rc = check_scan_chunks(m, probs, nullptr, 0);
  if (rc) return rc;
  if (!kfs || !sms) return cfail(m, BDLM_E_ARG, "null output arrays");
  Nccl *nc = nccl();
  const int W = m->world;
  const int n = probs[0].n;
  const int ef = bdlm_scan_elem_doubles(n, 0), eb = bdlm_scan_elem_doubles(n, 1);
  // Every device's phases are enqueued by its own host thread: local scan -> exchange -> finish,
  // forwards then backwards.  With peer mailboxes nothing on the host couples the devices (the
  // finish kernels wait on flags in device memory); with NCCL every thread issues the all-gather
  // of its own communicator rank.
  auto enqueue = [&](int i) -> int {
    Local &L = m->loc[i];
    int32_t *st = status ? status[i] : nullptr;
    unsigned long long *epoch_dev = L.flags + 2 * W;
    if (cudaSetDevice(L.device) != cudaSuccess) return BDLM_E_CUDA;  // worker threads start on device 0
    cudaError_t ce = launch_epoch_bump(epoch_dev, ctx_stream(L.ctx));
    if (ce != cudaSuccess) return BDLM_E_CUDA;
    for (int pass = 0; pass < 2; ++pass) {
      const int e = pass ? eb : ef;
      const ScanPeers *peers = m->peer ? &m->peers[pass] : nullptr;
      double *agg = L.agg + (size_t)pass * kMaxElem;
      double *aggs = L.aggs + (size_t)pass * W * kMaxElem;
      scan_set_peers(L.ctx, peers, epoch_dev);
      int rc = pass ? bdlm_scan_dist_backward_local(L.ctx, &probs[i], L.rank, W, &kfs[i], &sms[i], agg)
                    : bdlm_scan_dist_forward_local(L.ctx, &probs[i], L.rank, W, agg);
      if (!rc && !m->peer) {
        const int r = nc->AllGather(agg, aggs, (size_t)e, kNcclFloat64, L.nc, ctx_stream(L.ctx));
        if (r != 0) rc = BDLM_E_NCCL;
      }
      if (!rc)
        rc = pass ? bdlm_scan_dist_backward_finish(L.ctx, &probs[i], L.rank, W, aggs, &kfs[i], &sms[i], st)
                  : bdlm_scan_dist_forward_finish(L.ctx, &probs[i], L.rank, W, aggs, &kfs[i], st);
      scan_set_peers(L.ctx, nullptr, nullptr);
      if (rc) return rc;
    }
    return 0;
  };
  return for_each_local(m, enqueue);
}


// ---- the same long series' log-likelihoods and FFBS, cut along time over the ranks ---------------
int bdlm_comm_scan_loglik(bdlm_comm *m, const bdlm_problem *probs, double *const *m_last, double *const *C_last,
                          double *const *transition, double *const *innovations, int32_t *const *status) {
  int rc = check_scan_chunks(m, probs, nullptr, 0);
  if (rc) return rc;
  const int W = m->world, n = probs[0].n;
  const int ef = bdlm_scan_elem_doubles(n, 0), lp = bdlm_scan_dist_doubles(n, BDLM_SCAN_DIST_LOGLIK_PART);
  return for_each_local(m, [&](int i) -> int {
    const Local &L = m->loc[i];
    if (cudaSetDevice(L.device) != cudaSuccess) return BDLM_E_CUDA;  // worker threads start on device 0
    int r = bdlm_scan_dist_forward_local(L.ctx, &probs[i], L.rank, W, xch_send(L, 0));
    if (!r) r = xch_gather(L, W, 0, ef);
    if (!r) r = bdlm_scan_dist_loglik_partial(L.ctx, &probs[i], L.rank, W, xch_recv(L, W, 0), entry(m_last, i),
                                              entry(C_last, i), xch_send(L, 1));
    if (!r) r = xch_gather(L, W, 1, lp);
    if (!r) r = bdlm_scan_dist_loglik_finish(L.ctx, W, xch_recv(L, W, 1), entry(transition, i),
                                             entry(innovations, i), entry(status, i));
    return r;
  });
}

int bdlm_comm_scan_ffbs(bdlm_comm *m, const bdlm_problem *probs, const int64_t *first_row, int64_t total_T,
                        const double *const *z, double *const *theta, const bdlm_kf_out *kfs,
                        const bdlm_gibbs_stats *stats, int32_t *const *status) {
  if (m && (!first_row || !theta || !kfs)) return cfail(m, BDLM_E_ARG, "null first_row, theta or kfs array");
  int rc = check_scan_chunks(m, probs, first_row, total_T);
  if (rc) return rc;
  const int W = m->world, n = probs[0].n;
  const int ef = bdlm_scan_elem_doubles(n, 0), es = bdlm_scan_dist_doubles(n, BDLM_SCAN_DIST_SAMPLER_ELEM);
  const int fp = bdlm_scan_dist_doubles(n, BDLM_SCAN_DIST_FFBS_PART);
  return for_each_local(m, [&](int i) -> int {
    const Local &L = m->loc[i];
    if (cudaSetDevice(L.device) != cudaSuccess) return BDLM_E_CUDA;
    int32_t *st = entry(status, i);
    int r = bdlm_scan_dist_forward_local(L.ctx, &probs[i], L.rank, W, xch_send(L, 0));
    if (!r) r = xch_gather(L, W, 0, ef);
    if (!r) r = bdlm_scan_dist_ffbs_local(L.ctx, &probs[i], L.rank, W, first_row[i], total_T, xch_recv(L, W, 0),
                                          entry(z, i), theta[i], &kfs[i], xch_send(L, 1), st);
    if (!r) r = xch_gather(L, W, 1, es);
    if (!r) r = bdlm_scan_dist_ffbs_finish(L.ctx, &probs[i], L.rank, W, xch_recv(L, W, 1), theta[i], &kfs[i],
                                           xch_send(L, 2), st);
    if (!r) r = xch_gather(L, W, 2, fp);
    if (!r) r = bdlm_scan_dist_ffbs_stats_finish(L.ctx, n, W, xch_recv(L, W, 2), stats ? &stats[i] : nullptr, st);
    return r;
  });
}

int bdlm_comm_sync(bdlm_comm *m) {
  if (!m) return cfail(nullptr, BDLM_E_ARG, "null communicator");
  for (Local &L : m->loc) {
    int rc = bdlm_sync(L.ctx);
    if (rc) return cfail(m, rc, bdlm_last_error(L.ctx));
  }
  return 0;
}

}  // extern "C"
