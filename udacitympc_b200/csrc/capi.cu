// C ABI of libb200mpc.so (include/b200mpc.h): handles, device buffers, host<->device staging, multi-device
// sharding.  No CPU compute path exists here: every entry point launches the sm_100a kernels or fails.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <functional>
#include <memory>
#include <mutex>
#include <thread>
#include <fstream>
#include <new>
#include <sstream>
#include <string>
#include <vector>

#include "../../include/b200mpc.h"
#include "kernels.h"

using namespace b200mpc;

namespace {

thread_local std::string g_err;
int fail(int code, const std::string& msg) { g_err = msg; return code; }
int cuda_fail(cudaError_t e, const char* what) {
  return fail(B200MPC_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
#define CU(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return cuda_fail(e_, #x); } while (0)

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e == cudaSuccess) cap = bytes;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <class T> T* as() const { return (T*)p; }
};

}  // namespace

struct b200mpc_handle {
  Params P;
  SolveConfig cfg;
  SplitStreams ss;
  int device = 0;
  cudaStream_t stream = nullptr;
  DevBuf ws, in_aos, out_aos, traj_soa, traj_aos, obj, status, iters, misc0, misc3;
  DevBuf guess_aos, guess_soa, mult_soa, mult_aos;   // b200mpc_solve_batch_warm: x_init | mult_init rows and columns, mult
  DevBuf vjp_aos, vjp_soa, vjp_io;   // b200mpc_solve_batch_vjp: traj | mult | g_traj rows and columns, the per-problem rest
  bool timing_on = false;                                    // b200mpc_set_timing: measurement only, off by default
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> timing;   // around every solve while timing_on
  cudaEvent_t done = nullptr;   // recorded after every solve: the next solve on this handle (any stream) waits for it
  bool done_valid = false;
  b200mpc_params user_params;
  long long launches = 0;
  // CUDA graphs of whole solves (init + rounds x (factor, forward, step) + finisher), keyed by every launch argument
  struct GraphKey {
    int phase = 0, B = 0, steps = 0;   // phase: 0 whole solve, 1 bulk, 2 tail
    SolveIO io;
    const void *ws = nullptr, *tail = nullptr;   // the handle's workspace, the tail context of a pipelined solve
    int config_gen = 0;
  };
  struct GraphEntry {
    GraphKey key;
    cudaGraphExec_t exec;
    long long n_kernels;
  };
  std::vector<GraphEntry> graphs;
  bool use_graphs = true;
  // bumped by every setter that changes what a solve launches or the arguments it bakes in (part of the graph key)
  int config_gen = 0;
  // pipelined solves (b200mpc_set_pipeline): tail contexts, used round robin, and the events that order the calls
  static constexpr int kMaxPipe = 32;
  int pipe_depth = 0, pipe_slots = 0;
  DevBuf tail_ws;
  size_t tail_ctx_doubles = 0;          // of the allocation in tail_ws (pipe_depth contexts)
  int tail_ctx_N = 0, tail_ctx_slots = 0;
  cudaEvent_t main_free = nullptr, tail_free[kMaxPipe] = {};
  cudaStream_t tail_stream[kMaxPipe] = {};   // highest priority: the small kernels of a tail must not queue behind bulk blocks
  bool main_free_valid = false, tail_free_valid[kMaxPipe] = {};
  unsigned long long pipe_calls = 0;
};

namespace {

Params to_core(const b200mpc_params& p) {
  Params P;
  P.N = p.N; P.dt = p.dt; P.Lf = p.Lf; P.ref_v = p.ref_v;
  P.w_cte = p.w_cte; P.w_epsi = p.w_epsi; P.w_v = p.w_v; P.w_delta = p.w_delta; P.w_a = p.w_a;
  P.w_ddelta = p.w_ddelta; P.w_da = p.w_da; P.delta_max = p.delta_max; P.a_max = p.a_max;
  P.tol = p.tol; P.max_iter = p.max_iter;
  P.resto = 2;
  P.finalize();
  return P;
}

bool same_params(const b200mpc_params& a, const b200mpc_params& b) {
  return a.N == b.N && a.dt == b.dt && a.Lf == b.Lf && a.ref_v == b.ref_v && a.w_cte == b.w_cte && a.w_epsi == b.w_epsi &&
         a.w_v == b.w_v && a.w_delta == b.w_delta && a.w_a == b.w_a && a.w_ddelta == b.w_ddelta && a.w_da == b.w_da &&
         a.delta_max == b.delta_max && a.a_max == b.a_max && a.tol == b.tol && a.max_iter == b.max_iter;
}

int check_solve_args(const b200mpc_handle* h, int B, const void* st, const void* cf, int ncoef, const void* out8) {
  if (!h) return fail(B200MPC_ERR_ARG, "null handle");
  if (B < 0) return fail(B200MPC_ERR_ARG, "negative batch size");
  if (ncoef < 2 || ncoef > B200MPC_MAX_COEFFS) return fail(B200MPC_ERR_ARG, "ncoef must be in [2, 4] (polynomial degree 1..3)");
  if (B > 0 && (!st || !cf || !out8)) return fail(B200MPC_ERR_ARG, "null state6 / coeffs / out8");
  return 0;
}

int check_guess_args(const void* x_init, const void* mult_init, double mu_init) {
  if (mult_init && !x_init) return fail(B200MPC_ERR_ARG, "warm start: mult_init needs x_init");
  if (x_init && !(mu_init > 0.0 && mu_init <= 0.1)) return fail(B200MPC_ERR_ARG, "warm start: mu_init must be in (0, 0.1]");
  return 0;
}

bool same_key(const b200mpc_handle::GraphKey& a, const b200mpc_handle::GraphKey& b) {
  return a.phase == b.phase && a.B == b.B && a.steps == b.steps && a.io.state6 == b.io.state6 && a.io.coeffs == b.io.coeffs &&
         a.io.ncoef == b.io.ncoef && a.io.out8 == b.io.out8 && a.io.traj == b.io.traj && a.io.obj == b.io.obj &&
         a.io.status == b.io.status && a.io.iters == b.io.iters && a.io.io_aos == b.io.io_aos && a.io.x_init == b.io.x_init &&
         a.io.mult_init == b.io.mult_init && a.io.mu_init == b.io.mu_init && a.io.mult == b.io.mult && a.io.cost8 == b.io.cost8 &&
         a.io.model4 == b.io.model4 && a.ws == b.ws && a.tail == b.tail && a.config_gen == b.config_gen;
}

// One launch sequence (a whole solve, or one half of a pipelined one) on stream s.  One solve is ~85 dependent
// launches; replaying a captured graph keeps the host out of the inner loop (several ranks / streams per host otherwise
// become launch-bound).  The legacy default stream cannot be captured.
int run_solve(b200mpc_handle* h, const b200mpc_handle::GraphKey& key, cudaStream_t s, bool caller_captures,
              const std::function<cudaError_t(long long*)>& launch) {
  if (h->use_graphs && !caller_captures && s != nullptr && s != cudaStreamLegacy && s != cudaStreamPerThread) {
    b200mpc_handle::GraphEntry* hit = nullptr;
    for (auto& g : h->graphs)
      if (same_key(g.key, key)) hit = &g;
    if (!hit) {
      cudaGraph_t graph = nullptr;
      long long n = 0;
      if (cudaStreamBeginCapture(s, cudaStreamCaptureModeRelaxed) == cudaSuccess) {
        cudaError_t le = launch(&n);
        cudaError_t ce = cudaStreamEndCapture(s, &graph);
        if (le == cudaSuccess && ce == cudaSuccess && graph) {
          cudaGraphExec_t exec = nullptr;
          if (cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess) {
            if (h->graphs.size() >= 96) { cudaGraphExecDestroy(h->graphs.front().exec); h->graphs.erase(h->graphs.begin()); }
            h->graphs.push_back(b200mpc_handle::GraphEntry{key, exec, n});
            hit = &h->graphs.back();
          }
        }
        if (graph) cudaGraphDestroy(graph);
      }
      cudaGetLastError();   // a failed capture falls back to plain launches below
    }
    if (hit) {
      CU(cudaGraphLaunch(hit->exec, s));
      h->launches += hit->n_kernels;
      return 0;
    }
  }
  CU(launch(&h->launches));
  return 0;
}

// One solve on stream s.  The handle owns ONE workspace and one set of auxiliary streams, so solves on a handle are
// serialised on the device whatever streams the caller uses (an event recorded after each solve, waited for by the
// next).  With b200mpc_set_timing a pair of events brackets the solver kernels for bench.py.
int timed_solve(b200mpc_handle* h, int B, int steps, const SolveIO& io, cudaStream_t s) {
  // the caller may be capturing its stream into a graph of its own: then no nested capture, no external events
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (s != nullptr && s != cudaStreamLegacy) { if (cudaStreamIsCapturing(s, &cap) != cudaSuccess) { cudaGetLastError(); cap = cudaStreamCaptureStatusNone; } }
  const bool caller_captures = cap != cudaStreamCaptureStatusNone;
  if (caller_captures && h->ws.cap < solve_workspace_doubles(h->P.N, B) * sizeof(double))
    return fail(B200MPC_ERR_ARG, "the stream is being captured and the workspace would have to grow: run one solve of this size first");
  // Pipelined mode (b200mpc_set_pipeline): the solve is queued as bulk + tail, ordered against the neighbouring calls by
  // events instead of the one-solve-at-a-time rule below.
  const bool pipelined = h->pipe_depth > 0 && !caller_captures && steps == 1 && !h->cfg.warm_start && h->cfg.mode == kModePerPass &&
                         B >= h->cfg.fused_below && B > h->pipe_slots && h->cfg.compact_max_live > 0.0;
  if (h->ws.cap < solve_workspace_doubles(h->P.N, B) * sizeof(double) || !pipelined) {
    // a growing workspace, or a plain solve after pipelined ones: everything queued on this handle has to finish first
    for (int k = 0; k < h->pipe_depth; ++k)
      if (h->tail_free_valid[k]) CU(cudaStreamWaitEvent(s, h->tail_free[k], 0));
    if (h->main_free_valid) CU(cudaStreamWaitEvent(s, h->main_free, 0));
    if (h->ws.cap < solve_workspace_doubles(h->P.N, B) * sizeof(double) && h->pipe_calls) CU(cudaDeviceSynchronize());
  }
  CU(h->ws.ensure(solve_workspace_doubles(h->P.N, B) * sizeof(double)));
  b200mpc_handle::GraphKey key;   // what a graph of this call's launches bakes in
  key.B = B; key.steps = steps; key.io = io; key.ws = h->ws.p; key.config_gen = h->config_gen;
  if (pipelined) {
    const size_t ctx = solve_workspace_doubles(h->P.N, h->pipe_slots);
    if (h->tail_ctx_N != h->P.N || h->tail_ctx_slots != h->pipe_slots || h->tail_ws.cap < ctx * h->pipe_depth * sizeof(double)) {
      if (h->pipe_calls) CU(cudaDeviceSynchronize());
      CU(h->tail_ws.ensure(ctx * h->pipe_depth * sizeof(double)));
      h->tail_ctx_N = h->P.N; h->tail_ctx_slots = h->pipe_slots; h->tail_ctx_doubles = ctx;
    }
    const int k = (int)(h->pipe_calls++ % (unsigned long long)h->pipe_depth);
    TailCtx tail;
    tail.ws = h->tail_ws.as<double>() + (size_t)k * h->tail_ctx_doubles;
    tail.slots = h->pipe_slots;
    if (h->done_valid) { CU(cudaStreamWaitEvent(s, h->done, 0)); h->done_valid = false; }   // a plain solve queued before
    if (h->main_free_valid) CU(cudaStreamWaitEvent(s, h->main_free, 0));
    if (h->tail_free_valid[k]) CU(cudaStreamWaitEvent(s, h->tail_free[k], 0));
    key.phase = 1; key.tail = tail.ws;
    if (int rc = run_solve(h, key, s, false, [&](long long* n) { return launch_solve_bulk(h->P, B, io, h->ws.as<double>(), tail, h->cfg, s, n); })) return rc;
    CU(cudaEventRecord(h->main_free, s));
    h->main_free_valid = true;
    // the tail runs on the context's own high-priority stream, behind the bulk; the caller's stream then waits for it,
    // so the call stays stream-ordered for its caller
    cudaStream_t ts = h->tail_stream[k] ? h->tail_stream[k] : s;
    if (ts != s) CU(cudaStreamWaitEvent(ts, h->main_free, 0));
    key.phase = 2;
    if (int rc = run_solve(h, key, ts, false, [&](long long* n) { return launch_solve_tail(h->P, B, io, tail, h->cfg, ts, n); })) return rc;
    CU(cudaEventRecord(h->tail_free[k], ts));
    h->tail_free_valid[k] = true;
    if (ts != s) CU(cudaStreamWaitEvent(s, h->tail_free[k], 0));
    return 0;
  }
  if (!caller_captures && h->done_valid) CU(cudaStreamWaitEvent(s, h->done, 0));
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  const bool rec = h->timing_on && !caller_captures && h->timing.size() < 8192;
  if (rec) {
    CU(cudaEventCreate(&e0));
    if (cudaEventCreate(&e1) != cudaSuccess) { cudaEventDestroy(e0); return cuda_fail(cudaGetLastError(), "cudaEventCreate"); }
    cudaError_t e = cudaEventRecord(e0, s);
    if (e != cudaSuccess) { cudaEventDestroy(e0); cudaEventDestroy(e1); return cuda_fail(e, "cudaEventRecord"); }
  }
  int rc = run_solve(h, key, s, caller_captures,
                     [&](long long* n) { return launch_solve(h->P, B, steps, io, h->ws.as<double>(), h->cfg, s, &h->ss, n); });
  if (rec) {
    cudaError_t e = rc == 0 ? cudaEventRecord(e1, s) : cudaErrorUnknown;
    if (e == cudaSuccess) h->timing.emplace_back(e0, e1);
    else { cudaEventDestroy(e0); cudaEventDestroy(e1); if (rc == 0) rc = cuda_fail(e, "cudaEventRecord"); }
  }
  if (rc == 0 && !caller_captures) {
    CU(cudaEventRecord(h->done, s));
    h->done_valid = true;
  }
  return rc;
}

// One sensitivity launch (b200mpc_solve_batch_vjp*, b200mpc_solve_batch_jvp*) of B problems on stream s.  It uses the
// handle's workspace, so it is ordered like a plain solve in timed_solve: after everything queued on this handle,
// pipelined tails included, and before the next call.
int run_sens(b200mpc_handle* h, int B, cudaStream_t s, const std::function<cudaError_t(double*)>& launch) {
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (s != nullptr && s != cudaStreamLegacy) { if (cudaStreamIsCapturing(s, &cap) != cudaSuccess) { cudaGetLastError(); cap = cudaStreamCaptureStatusNone; } }
  const bool caller_captures = cap != cudaStreamCaptureStatusNone;
  const size_t need = solve_workspace_doubles(h->P.N, B) * sizeof(double);
  if (caller_captures && h->ws.cap < need)
    return fail(B200MPC_ERR_ARG, "the stream is being captured and the workspace would have to grow: run one solve of this size first");
  for (int k = 0; k < h->pipe_depth; ++k)
    if (h->tail_free_valid[k]) CU(cudaStreamWaitEvent(s, h->tail_free[k], 0));
  if (h->main_free_valid) CU(cudaStreamWaitEvent(s, h->main_free, 0));
  if (h->ws.cap < need && h->pipe_calls) CU(cudaDeviceSynchronize());
  CU(h->ws.ensure(need));
  if (!caller_captures && h->done_valid) CU(cudaStreamWaitEvent(s, h->done, 0));
  CU(launch(h->ws.as<double>()));
  h->launches += 1;
  if (!caller_captures) {
    CU(cudaEventRecord(h->done, s));
    h->done_valid = true;
  }
  return 0;
}
int run_vjp(b200mpc_handle* h, const VjpCostIO& io, cudaStream_t s) {
  return run_sens(h, io.B, s, [&](double* ws) { return launch_vjp(h->P, io, ws, s); });
}
int run_jvp(b200mpc_handle* h, const JvpIO& io, cudaStream_t s) {
  return run_sens(h, io.B, s, [&](double* ws) { return launch_jvp(h->P, io, ws, s); });
}

int check_vjp_args(const b200mpc_handle* h, int B, const void* st, const void* cf, int ncoef, const void* traj, const void* mult,
                   const void* g_out8, const void* g_traj, const void* g_obj) {
  if (!h) return fail(B200MPC_ERR_ARG, "null handle");
  if (B <= 0) return fail(B200MPC_ERR_ARG, "vjp: B must be positive");
  if (ncoef < 2 || ncoef > B200MPC_MAX_COEFFS) return fail(B200MPC_ERR_ARG, "ncoef must be in [2, 4] (polynomial degree 1..3)");
  if (!st || !cf || !traj || !mult) return fail(B200MPC_ERR_ARG, "vjp: null state6 / coeffs / traj / mult");
  if (!g_out8 && !g_traj && !g_obj) return fail(B200MPC_ERR_ARG, "vjp: no incoming gradient (g_out8, g_traj and g_obj are all null)");
  return 0;
}

int check_jvp_args(const b200mpc_handle* h, int B, const void* st, const void* cf, int ncoef, const void* traj, const void* mult,
                   const void* t_st, const void* t_cf, const void* t_c8, const void* t_m4) {
  if (!h) return fail(B200MPC_ERR_ARG, "null handle");
  if (B <= 0) return fail(B200MPC_ERR_ARG, "jvp: B must be positive");
  if (ncoef < 2 || ncoef > B200MPC_MAX_COEFFS) return fail(B200MPC_ERR_ARG, "ncoef must be in [2, 4] (polynomial degree 1..3)");
  if (!st || !cf || !traj || !mult) return fail(B200MPC_ERR_ARG, "jvp: null state6 / coeffs / traj / mult");
  if (!t_st && !t_cf && !t_c8 && !t_m4)
    return fail(B200MPC_ERR_ARG, "jvp: no tangent (t_state6, t_coeffs, t_cost8 and t_model4 are all null)");
  return 0;
}

}  // namespace

namespace {

// Persistent host threads for b200mpc_solve_batch_multi: one per extra device shard, created on first use and kept
// (a thread's first CUDA call costs about a millisecond of per-thread runtime set-up; a thread per call paid it every
// time).  Worker g queues and waits for shard g + 1 while the calling thread does shard 0.
struct Worker {
  std::thread th;
  std::mutex m;
  std::condition_variable cv;
  std::function<void()> task;
  bool has = false, quit = false;
  Worker() {
    th = std::thread([this]() {
      for (;;) {
        std::function<void()> t;
        {
          std::unique_lock<std::mutex> lk(m);
          cv.wait(lk, [this]() { return has || quit; });
          if (quit) return;
          t = std::move(task);
        }
        t();
        {
          std::lock_guard<std::mutex> lk(m);
          has = false;
        }
        cv.notify_all();
      }
    });
  }
  void start(std::function<void()> t) {
    {
      std::lock_guard<std::mutex> lk(m);
      task = std::move(t);
      has = true;
    }
    cv.notify_all();
  }
  void wait() {
    std::unique_lock<std::mutex> lk(m);
    cv.wait(lk, [this]() { return !has; });
  }
  ~Worker() {
    {
      std::lock_guard<std::mutex> lk(m);
      quit = true;
    }
    cv.notify_all();
    if (th.joinable()) th.join();
  }
};
std::mutex g_multi_mutex;                       // one multi call at a time uses the pool
std::vector<std::unique_ptr<Worker>> g_workers;

}  // namespace

extern "C" {

void b200mpc_default_params(b200mpc_params* p) {
  if (!p) return;
  p->N = 25; p->dt = 0.05; p->Lf = 2.67; p->ref_v = 40.0;
  p->w_cte = p->w_epsi = p->w_v = p->w_delta = p->w_a = p->w_ddelta = p->w_da = 1.0;
  p->delta_max = 0.436332; p->a_max = 1.0;
  p->tol = 1e-8; p->max_iter = 3000;
}

const char* b200mpc_last_error(void) { return g_err.c_str(); }

int b200mpc_create(const b200mpc_params* p, int device, b200mpc_handle** out) {
  if (!p || !out) return fail(B200MPC_ERR_ARG, "null params / out");
  if (p->N < 2 || p->N > 1024) return fail(B200MPC_ERR_ARG, "N must be in [2, 1024]");
  if (!(p->dt > 0) || !(p->Lf > 0) || !(p->delta_max > 0) || !(p->a_max > 0) || !(p->tol > 0) || p->max_iter < 0)
    return fail(B200MPC_ERR_ARG, "dt, Lf, delta_max, a_max, tol must be positive");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(B200MPC_ERR_CUDA, std::string("no CUDA device available (b200mpc has no CPU path): ") + cudaGetErrorString(e));
  if (device < 0 || device >= ndev) return fail(B200MPC_ERR_ARG, "device index out of range");
  CU(cudaSetDevice(device));
  CU(solver_prepare_device());
  b200mpc_handle* h = new (std::nothrow) b200mpc_handle();
  if (!h) return fail(B200MPC_ERR_NOMEM, "out of host memory");
  h->P = to_core(*p);
  h->user_params = *p;
  h->device = device;
  if (const char* e = getenv("B200MPC_NO_GRAPHS")) h->use_graphs = !(e[0] == '1');
  if (const char* e = getenv("B200MPC_NO_COOP")) h->cfg.coop = !(e[0] == '1');
  e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) { delete h; return cuda_fail(e, "cudaStreamCreate"); }
  e = cudaEventCreateWithFlags(&h->done, cudaEventDisableTiming);
  if (e != cudaSuccess) { cudaStreamDestroy(h->stream); delete h; return cuda_fail(e, "cudaEventCreate"); }
  for (int i = 0; i < 3; ++i) {   // auxiliary streams / events for the internal batch split
    if (cudaStreamCreateWithFlags(&h->ss.aux[i], cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ss.join[i], cudaEventDisableTiming) != cudaSuccess) break;
    h->ss.n_aux = i + 1;
  }
  if (cudaEventCreateWithFlags(&h->ss.fork, cudaEventDisableTiming) != cudaSuccess) h->ss.n_aux = 0;
  *out = h;
  return 0;
}

void b200mpc_destroy(b200mpc_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  for (auto& ev : h->timing) { cudaEventDestroy(ev.first); cudaEventDestroy(ev.second); }
  for (auto& g : h->graphs) cudaGraphExecDestroy(g.exec);
  for (int i = 0; i < 3; ++i) {
    if (h->ss.aux[i]) { cudaStreamSynchronize(h->ss.aux[i]); cudaStreamDestroy(h->ss.aux[i]); }
    if (h->ss.join[i]) cudaEventDestroy(h->ss.join[i]);
  }
  if (h->ss.fork) cudaEventDestroy(h->ss.fork);
  if (h->done) cudaEventDestroy(h->done);
  if (h->main_free) cudaEventDestroy(h->main_free);
  if (h->pipe_calls) cudaDeviceSynchronize();   // pipelined bulks ran on the callers' streams, tails on the handle's
  for (int k = 0; k < b200mpc_handle::kMaxPipe; ++k) {
    if (h->tail_free[k]) cudaEventDestroy(h->tail_free[k]);
    if (h->tail_stream[k]) cudaStreamDestroy(h->tail_stream[k]);
  }
  h->tail_ws.release();
  DevBuf* bufs[] = {&h->ws, &h->in_aos, &h->out_aos, &h->traj_soa, &h->traj_aos, &h->obj, &h->status, &h->iters, &h->misc0, &h->misc3,
                    &h->guess_aos, &h->guess_soa, &h->mult_soa, &h->mult_aos, &h->vjp_aos, &h->vjp_soa, &h->vjp_io};
  for (DevBuf* b : bufs) b->release();
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
}

int b200mpc_set_solver_mode(b200mpc_handle* h, int mode, int rounds, int fused_below) {
  if (!h) return fail(B200MPC_ERR_ARG, "null handle");
  if (mode != kModePerPass && mode != kModeFused) return fail(B200MPC_ERR_ARG, "mode must be 0 (per-pass kernels) or 1 (fused kernel)");
  if (rounds < 0 || rounds > 100000) return fail(B200MPC_ERR_ARG, "rounds out of range");
  h->cfg.mode = mode;
  if (rounds > 0) h->cfg.rounds = rounds;
  if (fused_below >= 0) h->cfg.fused_below = fused_below;
  ++h->config_gen;
  return 0;
}

int b200mpc_set_warm_start(b200mpc_handle* h, int enable, double mu_init) {
  if (!h) return fail(B200MPC_ERR_ARG, "null handle");
  if (enable && !(mu_init > 0.0 && mu_init <= 0.1)) return fail(B200MPC_ERR_ARG, "warm start: mu_init must be in (0, 0.1]");
  h->cfg.warm_start = enable != 0;
  if (enable) h->cfg.warm_mu = mu_init;
  ++h->config_gen;
  return 0;
}

int b200mpc_set_batch_split(b200mpc_handle* h, int parts) {
  if (!h) return fail(B200MPC_ERR_ARG, "null handle");
  if (parts < 1 || parts > 4) return fail(B200MPC_ERR_ARG, "batch split: parts must be 1..4");
  h->cfg.split = parts;
  ++h->config_gen;
  return 0;
}

int b200mpc_set_compaction(b200mpc_handle* h, double max_live_fraction, int from_round) {
  if (!h) return fail(B200MPC_ERR_ARG, "null handle");
  if (!(max_live_fraction >= 0.0 && max_live_fraction <= 1.0)) return fail(B200MPC_ERR_ARG, "compaction: max_live_fraction must be in [0, 1]");
  if (from_round < 1) return fail(B200MPC_ERR_ARG, "compaction: from_round must be >= 1");
  h->cfg.compact_max_live = max_live_fraction;
  h->cfg.compact_from = from_round;
  ++h->config_gen;
  return 0;
}

int b200mpc_set_handover(b200mpc_handle* h, int occupied_slots, int from_round) {
  if (!h) return fail(B200MPC_ERR_ARG, "null handle");
  if (occupied_slots < 0 || occupied_slots > (1 << 20)) return fail(B200MPC_ERR_ARG, "hand-over: occupied_slots must be in [0, 1048576]");
  if (from_round < 1) return fail(B200MPC_ERR_ARG, "hand-over: from_round must be >= 1");
  h->cfg.handover_below = occupied_slots;
  h->cfg.handover_from = from_round;
  ++h->config_gen;
  return 0;
}

int b200mpc_set_pipeline(b200mpc_handle* h, int depth, int tail_slots) {
  if (!h) return fail(B200MPC_ERR_ARG, "null handle");
  if (depth < 0 || depth > b200mpc_handle::kMaxPipe) return fail(B200MPC_ERR_ARG, "pipeline: depth must be in [0, 32]");
  if (depth > 0 && (tail_slots < 64 || tail_slots > (1 << 20))) return fail(B200MPC_ERR_ARG, "pipeline: tail_slots must be in [64, 1048576]");
  CU(cudaSetDevice(h->device));
  CU(cudaDeviceSynchronize());   // nothing of this handle is in flight while the contexts change
  int prio_lo = 0, prio_hi = 0;
  CU(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
  for (int k = 0; k < depth; ++k) {
    if (!h->tail_free[k]) CU(cudaEventCreateWithFlags(&h->tail_free[k], cudaEventDisableTiming));
    if (!h->tail_stream[k]) CU(cudaStreamCreateWithPriority(&h->tail_stream[k], cudaStreamNonBlocking, prio_hi));
  }
  if (depth > 0 && !h->main_free) CU(cudaEventCreateWithFlags(&h->main_free, cudaEventDisableTiming));
  for (int k = 0; k < b200mpc_handle::kMaxPipe; ++k) h->tail_free_valid[k] = false;
  h->main_free_valid = false;
  h->pipe_depth = depth;
  h->pipe_slots = depth > 0 ? (tail_slots + 63) / 64 * 64 : 0;
  h->pipe_calls = 0;
  ++h->config_gen;
  return 0;
}

int b200mpc_set_restoration(b200mpc_handle* h, int mode) {
  if (!h) return fail(B200MPC_ERR_ARG, "null handle");
  if (mode < 0 || mode > 2) return fail(B200MPC_ERR_ARG, "restoration: mode must be 0, 1 or 2");
  h->P.resto = mode;
  ++h->config_gen;
  return 0;
}

int b200mpc_num_vars(const b200mpc_handle* h) { return h ? 8 * h->P.N - 2 : 0; }
int b200mpc_num_mults(const b200mpc_handle* h) { return h ? 10 * h->P.N - 4 : 0; }
long long b200mpc_launch_count(const b200mpc_handle* h) { return h ? h->launches : 0; }

int b200mpc_solve_batch_device(b200mpc_handle* h, int B, const double* d_state6, const double* d_coeffs, int ncoef,
                               double* d_out8, double* d_traj, double* d_obj, int* d_status, int* d_iters,
                               void* stream) {
  return b200mpc_solve_batch_warm_device(h, B, d_state6, d_coeffs, ncoef, nullptr, nullptr, 0.0, d_out8, d_traj, nullptr, d_obj,
                                         d_status, d_iters, stream);
}

int b200mpc_solve_batch_warm_device(b200mpc_handle* h, int B, const double* d_state6, const double* d_coeffs, int ncoef,
                                    const double* d_x_init, const double* d_mult_init, double mu_init, double* d_out8,
                                    double* d_traj, double* d_mult, double* d_obj, int* d_status, int* d_iters, void* stream) {
  return b200mpc_solve_batch_cost_device(h, B, d_state6, d_coeffs, ncoef, nullptr, d_x_init, d_mult_init, mu_init, d_out8, d_traj,
                                         d_mult, d_obj, d_status, d_iters, stream);
}

int b200mpc_solve_batch_cost_device(b200mpc_handle* h, int B, const double* d_state6, const double* d_coeffs, int ncoef,
                                    const double* d_cost8, const double* d_x_init, const double* d_mult_init, double mu_init,
                                    double* d_out8, double* d_traj, double* d_mult, double* d_obj, int* d_status, int* d_iters,
                                    void* stream) {
  return b200mpc_solve_batch_model_device(h, B, d_state6, d_coeffs, ncoef, d_cost8, nullptr, d_x_init, d_mult_init, mu_init, d_out8,
                                          d_traj, d_mult, d_obj, d_status, d_iters, stream);
}

int b200mpc_solve_batch_model_device(b200mpc_handle* h, int B, const double* d_state6, const double* d_coeffs, int ncoef,
                                     const double* d_cost8, const double* d_model4, const double* d_x_init,
                                     const double* d_mult_init, double mu_init, double* d_out8, double* d_traj, double* d_mult,
                                     double* d_obj, int* d_status, int* d_iters, void* stream) {
  if (int rc = check_solve_args(h, B, d_state6, d_coeffs, ncoef, d_out8)) return rc;
  if (int rc = check_guess_args(d_x_init, d_mult_init, mu_init)) return rc;
  if (B == 0) return 0;
  CU(cudaSetDevice(h->device));
  SolveIO io;
  io.state6 = d_state6; io.coeffs = d_coeffs; io.ncoef = ncoef;
  io.out8 = d_out8; io.traj = d_traj; io.obj = d_obj; io.status = d_status; io.iters = d_iters;
  io.x_init = d_x_init; io.mult_init = d_mult_init; io.mu_init = d_x_init ? mu_init : 0.0; io.mult = d_mult;
  io.cost8 = d_cost8; io.model4 = d_model4;
  return timed_solve(h, B, 1, io, stream ? (cudaStream_t)stream : h->stream);
}

// queues the copy of the host arrays state6 [B][6], coeffs [B][ncoef], cost8 [B][8] and model4 [B][4] (if given) to
// in_aos and points io's inputs there (io_aos = 1)
static int stage_inputs(b200mpc_handle* h, int B, const double* state6, const double* coeffs, int ncoef, SolveIO* io,
                        const double* cost8 = nullptr, const double* model4 = nullptr) {
  const size_t nb = (size_t)B;
  CU(h->in_aos.ensure(nb * (6 + ncoef + (cost8 ? 8 : 0) + (model4 ? 4 : 0)) * sizeof(double)));
  double* d_st = h->in_aos.as<double>();
  double* d_cf = d_st + nb * 6;
  CU(cudaMemcpyAsync(d_st, state6, nb * 6 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(d_cf, coeffs, nb * ncoef * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  io->state6 = d_st; io->coeffs = d_cf; io->ncoef = ncoef; io->io_aos = 1;
  if (cost8) {
    double* d_c8 = d_cf + nb * ncoef;
    CU(cudaMemcpyAsync(d_c8, cost8, nb * 8 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    io->cost8 = d_c8;
  }
  if (model4) {
    double* d_m4 = d_cf + nb * (ncoef + (cost8 ? 8 : 0));
    CU(cudaMemcpyAsync(d_m4, model4, nb * 4 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    io->model4 = d_m4;
  }
  return 0;
}

// Everything b200mpc_solve_batch does except the final wait: copies, solve and copies back are queued on the handle's
// stream (asynchronous when the host buffers are pinned).
// x_init / mult_init / mult (b200mpc_solve_batch_warm): per-problem rows on the host, moved through the tiled transposes
// like traj.  cost8 / model4 (b200mpc_solve_batch_model): per-problem rows, read by the kernels in that layout.
static int enqueue_solve_batch(b200mpc_handle* h, int B, const double* state6, const double* coeffs, int ncoef, double* out8,
                               double* traj, double* obj, int* status, int* iters, const double* x_init = nullptr,
                               const double* mult_init = nullptr, double mu_init = 0.0, double* mult = nullptr,
                               const double* cost8 = nullptr, const double* model4 = nullptr) {
  if (int rc = check_solve_args(h, B, state6, coeffs, ncoef, out8)) return rc;
  if (int rc = check_guess_args(x_init, mult_init, mu_init)) return rc;
  if (B == 0) return 0;
  CU(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  const int nv = 8 * h->P.N - 2;
  const size_t nb = (size_t)B;
  // stage: H2D -> solve -> D2H.  The solver kernels read state6 / coeffs and write out8 in the reference's per-problem
  // order themselves (io_aos = 1: K6 fused into init / write_result); only the optional full trajectory goes through the
  // tiled transpose.
  CU(h->out_aos.ensure(nb * 8 * sizeof(double)));
  CU(h->obj.ensure(nb * sizeof(double)));
  CU(h->status.ensure(nb * sizeof(int)));
  CU(h->iters.ensure(nb * sizeof(int)));
  if (traj) { CU(h->traj_soa.ensure(nb * nv * sizeof(double))); CU(h->traj_aos.ensure(nb * nv * sizeof(double))); }
  SolveIO io;
  if (int rc = stage_inputs(h, B, state6, coeffs, ncoef, &io, cost8, model4)) return rc;
  io.out8 = h->out_aos.as<double>(); io.traj = traj ? h->traj_soa.as<double>() : nullptr;
  io.obj = h->obj.as<double>(); io.status = h->status.as<int>(); io.iters = h->iters.as<int>();
  const int nm = 10 * h->P.N - 4;
  if (x_init) {
    const size_t n = nb * (nv + (mult_init ? nm : 0));
    CU(h->guess_aos.ensure(n * sizeof(double)));
    CU(h->guess_soa.ensure(n * sizeof(double)));
    double *ga = h->guess_aos.as<double>(), *gs = h->guess_soa.as<double>();
    CU(cudaMemcpyAsync(ga, x_init, nb * nv * sizeof(double), cudaMemcpyHostToDevice, s));
    CU(launch_aos_to_soa(ga, gs, B, nv, s));
    h->launches += 1;
    io.x_init = gs; io.mu_init = mu_init;
    if (mult_init) {
      CU(cudaMemcpyAsync(ga + nb * nv, mult_init, nb * nm * sizeof(double), cudaMemcpyHostToDevice, s));
      CU(launch_aos_to_soa(ga + nb * nv, gs + nb * nv, B, nm, s));
      h->launches += 1;
      io.mult_init = gs + nb * nv;
    }
  }
  if (mult) {
    CU(h->mult_soa.ensure(nb * nm * sizeof(double)));
    CU(h->mult_aos.ensure(nb * nm * sizeof(double)));
    io.mult = h->mult_soa.as<double>();
  }
  if (int rc = timed_solve(h, B, 1, io, s)) return rc;
  CU(cudaMemcpyAsync(out8, h->out_aos.p, nb * 8 * sizeof(double), cudaMemcpyDeviceToHost, s));
  if (traj) {
    CU(launch_soa_to_aos(h->traj_soa.as<double>(), h->traj_aos.as<double>(), B, nv, s));
    h->launches += 1;
    CU(cudaMemcpyAsync(traj, h->traj_aos.p, nb * nv * sizeof(double), cudaMemcpyDeviceToHost, s));
  }
  if (mult) {
    CU(launch_soa_to_aos(h->mult_soa.as<double>(), h->mult_aos.as<double>(), B, nm, s));
    h->launches += 1;
    CU(cudaMemcpyAsync(mult, h->mult_aos.p, nb * nm * sizeof(double), cudaMemcpyDeviceToHost, s));
  }
  if (obj) CU(cudaMemcpyAsync(obj, h->obj.p, nb * sizeof(double), cudaMemcpyDeviceToHost, s));
  if (status) CU(cudaMemcpyAsync(status, h->status.p, nb * sizeof(int), cudaMemcpyDeviceToHost, s));
  if (iters) CU(cudaMemcpyAsync(iters, h->iters.p, nb * sizeof(int), cudaMemcpyDeviceToHost, s));
  return 0;
}

int b200mpc_solve_batch(b200mpc_handle* h, int B, const double* state6, const double* coeffs, int ncoef, double* out8,
                        double* traj, double* obj, int* status, int* iters) {
  if (int rc = enqueue_solve_batch(h, B, state6, coeffs, ncoef, out8, traj, obj, status, iters)) return rc;
  if (B == 0) return 0;
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

int b200mpc_solve_batch_warm(b200mpc_handle* h, int B, const double* state6, const double* coeffs, int ncoef,
                             const double* x_init, const double* mult_init, double mu_init, double* out8, double* traj,
                             double* mult, double* obj, int* status, int* iters) {
  return b200mpc_solve_batch_cost(h, B, state6, coeffs, ncoef, nullptr, x_init, mult_init, mu_init, out8, traj, mult, obj, status,
                                  iters);
}

int b200mpc_solve_batch_cost(b200mpc_handle* h, int B, const double* state6, const double* coeffs, int ncoef, const double* cost8,
                             const double* x_init, const double* mult_init, double mu_init, double* out8, double* traj,
                             double* mult, double* obj, int* status, int* iters) {
  return b200mpc_solve_batch_model(h, B, state6, coeffs, ncoef, cost8, nullptr, x_init, mult_init, mu_init, out8, traj, mult, obj,
                                   status, iters);
}

int b200mpc_solve_batch_model(b200mpc_handle* h, int B, const double* state6, const double* coeffs, int ncoef, const double* cost8,
                              const double* model4, const double* x_init, const double* mult_init, double mu_init, double* out8,
                              double* traj, double* mult, double* obj, int* status, int* iters) {
  if (int rc = enqueue_solve_batch(h, B, state6, coeffs, ncoef, out8, traj, obj, status, iters, x_init, mult_init, mu_init, mult,
                                   cost8, model4))
    return rc;
  if (B == 0) return 0;
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

int b200mpc_solve_batch_vjp_device(b200mpc_handle* h, int B, const double* d_state6, const double* d_coeffs, int ncoef,
                                   const double* d_traj, const double* d_mult, const double* d_g_out8, const double* d_g_traj,
                                   const double* d_g_obj, double* d_grad_state6, double* d_grad_coeffs, double* d_grad_params,
                                   int* d_status, void* stream) {
  return b200mpc_solve_batch_vjp_cost_device(h, B, d_state6, d_coeffs, ncoef, nullptr, d_traj, d_mult, d_g_out8, d_g_traj, d_g_obj,
                                             d_grad_state6, d_grad_coeffs, d_grad_params, d_status, stream);
}

int b200mpc_solve_batch_vjp_cost_device(b200mpc_handle* h, int B, const double* d_state6, const double* d_coeffs, int ncoef,
                                        const double* d_cost8, const double* d_traj, const double* d_mult, const double* d_g_out8,
                                        const double* d_g_traj, const double* d_g_obj, double* d_grad_state6, double* d_grad_coeffs,
                                        double* d_grad_params, int* d_status, void* stream) {
  return b200mpc_solve_batch_vjp_model_device(h, B, d_state6, d_coeffs, ncoef, d_cost8, nullptr, d_traj, d_mult, d_g_out8, d_g_traj,
                                              d_g_obj, d_grad_state6, d_grad_coeffs, d_grad_params, nullptr, d_status, stream);
}

int b200mpc_solve_batch_vjp_model_device(b200mpc_handle* h, int B, const double* d_state6, const double* d_coeffs, int ncoef,
                                         const double* d_cost8, const double* d_model4, const double* d_traj, const double* d_mult,
                                         const double* d_g_out8, const double* d_g_traj, const double* d_g_obj,
                                         double* d_grad_state6, double* d_grad_coeffs, double* d_grad_params,
                                         double* d_grad_model, int* d_status, void* stream) {
  if (int rc = check_vjp_args(h, B, d_state6, d_coeffs, ncoef, d_traj, d_mult, d_g_out8, d_g_traj, d_g_obj)) return rc;
  CU(cudaSetDevice(h->device));
  VjpCostIO io;
  io.B = B; io.ncoef = ncoef; io.io_aos = 0; io.cost8 = d_cost8; io.model4 = d_model4; io.grad_model = d_grad_model;
  io.state6 = d_state6; io.coeffs = d_coeffs; io.traj = d_traj; io.mult = d_mult;
  io.g_out8 = d_g_out8; io.g_traj = d_g_traj; io.g_obj = d_g_obj;
  io.grad_state6 = d_grad_state6; io.grad_coeffs = d_grad_coeffs; io.grad_params = d_grad_params; io.status = d_status;
  return run_vjp(h, io, stream ? (cudaStream_t)stream : h->stream);
}

// Host buffers: state6 / coeffs / g_out8 / g_obj and the outputs are read and written per problem by the kernel (io_aos = 1);
// traj / mult / g_traj go through the tiled transposes.
int b200mpc_solve_batch_vjp(b200mpc_handle* h, int B, const double* state6, const double* coeffs, int ncoef, const double* traj,
                            const double* mult, const double* g_out8, const double* g_traj, const double* g_obj,
                            double* grad_state6, double* grad_coeffs, double* grad_params, int* status) {
  return b200mpc_solve_batch_vjp_cost(h, B, state6, coeffs, ncoef, nullptr, traj, mult, g_out8, g_traj, g_obj, grad_state6,
                                      grad_coeffs, grad_params, status);
}

int b200mpc_solve_batch_vjp_cost(b200mpc_handle* h, int B, const double* state6, const double* coeffs, int ncoef, const double* cost8,
                                 const double* traj, const double* mult, const double* g_out8, const double* g_traj,
                                 const double* g_obj, double* grad_state6, double* grad_coeffs, double* grad_params, int* status) {
  return b200mpc_solve_batch_vjp_model(h, B, state6, coeffs, ncoef, cost8, nullptr, traj, mult, g_out8, g_traj, g_obj, grad_state6,
                                       grad_coeffs, grad_params, nullptr, status);
}

int b200mpc_solve_batch_vjp_model(b200mpc_handle* h, int B, const double* state6, const double* coeffs, int ncoef, const double* cost8,
                                  const double* model4, const double* traj, const double* mult, const double* g_out8,
                                  const double* g_traj, const double* g_obj, double* grad_state6, double* grad_coeffs,
                                  double* grad_params, double* grad_model, int* status) {
  if (int rc = check_vjp_args(h, B, state6, coeffs, ncoef, traj, mult, g_out8, g_traj, g_obj)) return rc;
  CU(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  const size_t nb = (size_t)B, nv = 8 * (size_t)h->P.N - 2, nm = 10 * (size_t)h->P.N - 4;
  const size_t nrows = nv + nm + (g_traj ? nv : 0);
  CU(h->vjp_aos.ensure(nb * nrows * sizeof(double)));
  CU(h->vjp_soa.ensure(nb * nrows * sizeof(double)));
  // per problem: g_out8 (8) | g_obj (1) | grad_state6 (6) | grad_coeffs (ncoef) | grad_params (8) | grad_model (4, if asked)
  CU(h->vjp_io.ensure(nb * (23 + ncoef + (grad_model ? 4 : 0)) * sizeof(double)));
  CU(h->status.ensure(nb * sizeof(int)));
  SolveIO in;
  if (int rc = stage_inputs(h, B, state6, coeffs, ncoef, &in, cost8, model4)) return rc;
  double *ga = h->vjp_aos.as<double>(), *gs = h->vjp_soa.as<double>(), *d = h->vjp_io.as<double>();
  const double* rows[3] = {traj, mult, g_traj};
  const size_t len[3] = {nv, nm, nv};
  size_t off = 0;
  for (int i = 0; i < 3; ++i) {
    if (!rows[i]) continue;
    CU(cudaMemcpyAsync(ga + nb * off, rows[i], nb * len[i] * sizeof(double), cudaMemcpyHostToDevice, s));
    CU(launch_aos_to_soa(ga + nb * off, gs + nb * off, B, (int)len[i], s));
    h->launches += 1;
    off += len[i];
  }
  if (g_out8) CU(cudaMemcpyAsync(d, g_out8, nb * 8 * sizeof(double), cudaMemcpyHostToDevice, s));
  if (g_obj) CU(cudaMemcpyAsync(d + nb * 8, g_obj, nb * sizeof(double), cudaMemcpyHostToDevice, s));
  VjpCostIO io;
  io.B = B; io.ncoef = ncoef; io.io_aos = 1; io.cost8 = in.cost8; io.model4 = in.model4;
  io.state6 = in.state6; io.coeffs = in.coeffs; io.traj = gs; io.mult = gs + nb * nv;
  io.g_out8 = g_out8 ? d : nullptr; io.g_traj = g_traj ? gs + nb * (nv + nm) : nullptr; io.g_obj = g_obj ? d + nb * 8 : nullptr;
  io.grad_state6 = d + nb * 9; io.grad_coeffs = d + nb * 15; io.grad_params = d + nb * (15 + ncoef);
  io.grad_model = grad_model ? d + nb * (23 + ncoef) : nullptr;
  io.status = h->status.as<int>();
  if (int rc = run_vjp(h, io, s)) return rc;
  if (grad_state6) CU(cudaMemcpyAsync(grad_state6, io.grad_state6, nb * 6 * sizeof(double), cudaMemcpyDeviceToHost, s));
  if (grad_coeffs) CU(cudaMemcpyAsync(grad_coeffs, io.grad_coeffs, nb * ncoef * sizeof(double), cudaMemcpyDeviceToHost, s));
  if (grad_params) CU(cudaMemcpyAsync(grad_params, io.grad_params, nb * 8 * sizeof(double), cudaMemcpyDeviceToHost, s));
  if (grad_model) CU(cudaMemcpyAsync(grad_model, io.grad_model, nb * 4 * sizeof(double), cudaMemcpyDeviceToHost, s));
  if (status) CU(cudaMemcpyAsync(status, h->status.p, nb * sizeof(int), cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  return 0;
}

int b200mpc_solve_batch_jvp_device(b200mpc_handle* h, int B, const double* d_state6, const double* d_coeffs, int ncoef,
                                   const double* d_cost8, const double* d_model4, const double* d_traj, const double* d_mult,
                                   const double* d_t_state6, const double* d_t_coeffs, const double* d_t_cost8,
                                   const double* d_t_model4, double* d_t_out8, double* d_t_traj, double* d_t_obj, int* d_status,
                                   void* stream) {
  if (int rc = check_jvp_args(h, B, d_state6, d_coeffs, ncoef, d_traj, d_mult, d_t_state6, d_t_coeffs, d_t_cost8, d_t_model4))
    return rc;
  CU(cudaSetDevice(h->device));
  JvpIO io;
  io.B = B; io.ncoef = ncoef; io.io_aos = 0;
  io.state6 = d_state6; io.coeffs = d_coeffs; io.cost8 = d_cost8; io.model4 = d_model4; io.traj = d_traj; io.mult = d_mult;
  io.t_state6 = d_t_state6; io.t_coeffs = d_t_coeffs; io.t_cost8 = d_t_cost8; io.t_model4 = d_t_model4;
  io.t_out8 = d_t_out8; io.t_traj = d_t_traj; io.t_obj = d_t_obj; io.status = d_status;
  return run_jvp(h, io, stream ? (cudaStream_t)stream : h->stream);
}

// Host buffers: the per-problem inputs, their tangents and t_out8 / t_obj are read and written per problem by the kernel
// (io_aos = 1); traj / mult go in and t_traj comes out through the tiled transposes.
int b200mpc_solve_batch_jvp(b200mpc_handle* h, int B, const double* state6, const double* coeffs, int ncoef, const double* cost8,
                            const double* model4, const double* traj, const double* mult, const double* t_state6,
                            const double* t_coeffs, const double* t_cost8, const double* t_model4, double* t_out8,
                            double* t_traj, double* t_obj, int* status) {
  if (int rc = check_jvp_args(h, B, state6, coeffs, ncoef, traj, mult, t_state6, t_coeffs, t_cost8, t_model4)) return rc;
  CU(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  const size_t nb = (size_t)B, nv = 8 * (size_t)h->P.N - 2, nm = 10 * (size_t)h->P.N - 4;
  // rows: traj | mult in, then t_traj out (its transpose reuses the input rows, which are consumed by then)
  CU(h->vjp_aos.ensure(nb * (nv + nm) * sizeof(double)));
  CU(h->vjp_soa.ensure(nb * (nv + nm + (t_traj ? nv : 0)) * sizeof(double)));
  // per problem: t_state6 (6) | t_coeffs (ncoef) | t_cost8 (8) | t_model4 (4) | t_out8 (8) | t_obj (1)
  CU(h->vjp_io.ensure(nb * (27 + ncoef) * sizeof(double)));
  CU(h->status.ensure(nb * sizeof(int)));
  SolveIO in;
  if (int rc = stage_inputs(h, B, state6, coeffs, ncoef, &in, cost8, model4)) return rc;
  double *ga = h->vjp_aos.as<double>(), *gs = h->vjp_soa.as<double>(), *d = h->vjp_io.as<double>();
  CU(cudaMemcpyAsync(ga, traj, nb * nv * sizeof(double), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(ga + nb * nv, mult, nb * nm * sizeof(double), cudaMemcpyHostToDevice, s));
  CU(launch_aos_to_soa(ga, gs, B, (int)nv, s));
  CU(launch_aos_to_soa(ga + nb * nv, gs + nb * nv, B, (int)nm, s));
  h->launches += 2;
  const double* tin[4] = {t_state6, t_coeffs, t_cost8, t_model4};
  const size_t tlen[4] = {6, (size_t)ncoef, 8, 4};
  const double* tdev[4] = {nullptr, nullptr, nullptr, nullptr};
  size_t off = 0;
  for (int i = 0; i < 4; ++i) {
    if (tin[i]) {
      CU(cudaMemcpyAsync(d + nb * off, tin[i], nb * tlen[i] * sizeof(double), cudaMemcpyHostToDevice, s));
      tdev[i] = d + nb * off;
    }
    off += tlen[i];
  }
  JvpIO io;
  io.B = B; io.ncoef = ncoef; io.io_aos = 1;
  io.state6 = in.state6; io.coeffs = in.coeffs; io.cost8 = in.cost8; io.model4 = in.model4; io.traj = gs; io.mult = gs + nb * nv;
  io.t_state6 = tdev[0]; io.t_coeffs = tdev[1]; io.t_cost8 = tdev[2]; io.t_model4 = tdev[3];
  io.t_out8 = d + nb * off; io.t_obj = d + nb * (off + 8); io.t_traj = t_traj ? gs + nb * (nv + nm) : nullptr;
  io.status = h->status.as<int>();
  if (int rc = run_jvp(h, io, s)) return rc;
  if (t_traj) {
    CU(launch_soa_to_aos(io.t_traj, ga, B, (int)nv, s));
    h->launches += 1;
    CU(cudaMemcpyAsync(t_traj, ga, nb * nv * sizeof(double), cudaMemcpyDeviceToHost, s));
  }
  if (t_out8) CU(cudaMemcpyAsync(t_out8, io.t_out8, nb * 8 * sizeof(double), cudaMemcpyDeviceToHost, s));
  if (t_obj) CU(cudaMemcpyAsync(t_obj, io.t_obj, nb * sizeof(double), cudaMemcpyDeviceToHost, s));
  if (status) CU(cudaMemcpyAsync(status, h->status.p, nb * sizeof(int), cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  return 0;
}

int b200mpc_solve_batch_async(b200mpc_handle* h, int B, const double* state6, const double* coeffs, int ncoef, double* out8,
                              double* traj, double* obj, int* status, int* iters) {
  return enqueue_solve_batch(h, B, state6, coeffs, ncoef, out8, traj, obj, status, iters);
}

int b200mpc_wait(b200mpc_handle* h) {
  if (!h) return fail(B200MPC_ERR_ARG, "null handle");
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

int b200mpc_solve_batch_multi(b200mpc_handle* const* hs, int n_handles, int B, const double* state6,
                              const double* coeffs, int ncoef, double* out8, double* traj, double* obj, int* status,
                              int* iters) {
  if (!hs || n_handles <= 0) return fail(B200MPC_ERR_ARG, "no handles");
  for (int g = 0; g < n_handles; ++g)
    if (!hs[g]) return fail(B200MPC_ERR_ARG, "null handle in list");
  if (B < 0) return fail(B200MPC_ERR_ARG, "negative batch size");
  // the shards write rows of one result array: same horizon / parameters everywhere, and no handle twice (two host
  // threads would share one workspace and stream)
  for (int g = 0; g < n_handles; ++g) {
    for (int k = 0; k < g; ++k)
      if (hs[k] == hs[g]) return fail(B200MPC_ERR_ARG, "handle " + std::to_string(g) + " repeats handle " + std::to_string(k));
    if (!same_params(hs[g]->user_params, hs[0]->user_params) || hs[g]->P.resto != hs[0]->P.resto)
      return fail(B200MPC_ERR_ARG, "handle " + std::to_string(g) + " was created with other parameters than handle 0");
  }
  if (int rc0 = check_solve_args(hs[0], B, state6, coeffs, ncoef, out8)) return rc0;
  if (B == 0) return 0;
  // Shard g is queued (copies in, solve graph, copies out: all asynchronous on the handle's stream) and waited for by
  // its own persistent host thread, shard 0 by the calling thread, so the devices start within microseconds of each
  // other.  (Pageable host buffers make the copies synchronous; the shards still overlap, one thread each.)
  const int nv = 8 * hs[0]->P.N - 2;
  std::lock_guard<std::mutex> pool_lock(g_multi_mutex);
  while ((int)g_workers.size() < n_handles - 1) g_workers.emplace_back(new Worker());
  std::vector<int> rc(n_handles, 0);
  std::vector<std::string> msg(n_handles);
  auto shard = [&](int g) {
    // contiguous index ranges, remainder to the last device (SURVEY 8e)
    const long long lo = (long long)B / n_handles * g;
    const long long hi = g == n_handles - 1 ? B : (long long)B / n_handles * (g + 1);
    rc[g] = b200mpc_solve_batch(hs[g], (int)(hi - lo), state6 + lo * 6, coeffs + lo * ncoef, ncoef, out8 + lo * 8,
                                traj ? traj + lo * nv : nullptr, obj ? obj + lo : nullptr, status ? status + lo : nullptr,
                                iters ? iters + lo : nullptr);
    if (rc[g]) msg[g] = b200mpc_last_error();   // thread-local: read on the thread that failed
  };
  for (int g = 1; g < n_handles; ++g) g_workers[g - 1]->start([&shard, g]() { shard(g); });
  shard(0);
  for (int g = 1; g < n_handles; ++g) g_workers[g - 1]->wait();
  for (int g = 0; g < n_handles; ++g)
    if (rc[g]) return fail(rc[g], "device shard " + std::to_string(g) + ": " + msg[g]);
  return 0;
}

int b200mpc_closed_loop_batch(b200mpc_handle* h, int B, int steps, const double* state6, const double* coeffs,
                              int ncoef, double* hist8, double* cost, int* iters) {
  if (int rc = check_solve_args(h, B, state6, coeffs, ncoef, hist8)) return rc;
  if (steps < 1) return fail(B200MPC_ERR_ARG, "steps must be >= 1");
  if (B == 0) return 0;
  CU(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  const size_t nb = (size_t)B, ns = (size_t)steps;
  CU(h->out_aos.ensure(ns * nb * 8 * sizeof(double)));
  CU(h->obj.ensure(ns * nb * sizeof(double)));
  CU(h->iters.ensure(ns * nb * sizeof(int)));
  SolveIO io;
  if (int rc = stage_inputs(h, B, state6, coeffs, ncoef, &io)) return rc;
  // every step's 8-vector is written as [B][8] rows by the solver kernels (and read back as the next initial state)
  io.out8 = h->out_aos.as<double>(); io.obj = h->obj.as<double>(); io.iters = h->iters.as<int>();
  if (int rc = timed_solve(h, B, steps, io, s)) return rc;
  CU(cudaMemcpyAsync(hist8, h->out_aos.p, ns * nb * 8 * sizeof(double), cudaMemcpyDeviceToHost, s));
  if (cost) CU(cudaMemcpyAsync(cost, h->obj.p, ns * nb * sizeof(double), cudaMemcpyDeviceToHost, s));
  if (iters) CU(cudaMemcpyAsync(iters, h->iters.p, ns * nb * sizeof(int), cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  return 0;
}

// ------------------------------------------------------------------------------------------------
static int check_fit_args(const b200mpc_handle* h, int B, const void* xs, const void* ys, int m, int order, const void* out) {
  if (!h) return fail(B200MPC_ERR_ARG, "null handle");
  if (B < 0) return fail(B200MPC_ERR_ARG, "negative batch size");
  if (m < 2 || m > B200MPC_MAX_FIT_POINTS) return fail(B200MPC_ERR_ARG, "polyfit: m must be in [2, 16]");
  if (!(order >= 1 && order <= m - 1)) return fail(B200MPC_ERR_ARG, "polyfit: requires 1 <= order <= m-1 (helpers.h:26)");
  if (order > B200MPC_MAX_FIT_ORDER) return fail(B200MPC_ERR_ARG, "polyfit: order must be <= 7");
  if (B > 0 && (!xs || !ys || !out)) return fail(B200MPC_ERR_ARG, "null xs / ys / coeffs_out");
  return 0;
}

int b200mpc_polyfit_batch_device(b200mpc_handle* h, int B, const double* d_xs, const double* d_ys, int m, int order,
                                 double* d_coeffs_out, void* stream) {
  if (int rc = check_fit_args(h, B, d_xs, d_ys, m, order, d_coeffs_out)) return rc;
  if (B == 0) return 0;
  CU(cudaSetDevice(h->device));
  CU(launch_polyfit(d_xs, d_ys, B, m, order, d_coeffs_out, stream ? (cudaStream_t)stream : h->stream));
  h->launches += 1;
  return 0;
}

int b200mpc_polyfit_batch(b200mpc_handle* h, int B, const double* xs, const double* ys, int m, int order,
                          double* coeffs_out) {
  if (int rc = check_fit_args(h, B, xs, ys, m, order, coeffs_out)) return rc;
  if (B == 0) return 0;
  CU(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  const size_t nb = (size_t)B;
  const int n = order + 1;
  CU(h->misc0.ensure(nb * 2 * m * sizeof(double)));   // xs | ys, per-fit rows as the caller has them
  CU(h->misc3.ensure(nb * n * sizeof(double)));       // coefficient rows
  double* a = h->misc0.as<double>();
  CU(cudaMemcpyAsync(a, xs, nb * m * sizeof(double), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(a + nb * m, ys, nb * m * sizeof(double), cudaMemcpyHostToDevice, s));
  CU(launch_polyfit(a, a + nb * m, B, m, order, h->misc3.as<double>(), s, 1));
  h->launches += 1;
  CU(cudaMemcpyAsync(coeffs_out, h->misc3.p, nb * n * sizeof(double), cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  return 0;
}

int b200mpc_polyeval_batch_device(b200mpc_handle* h, int B, const double* d_coeffs, int ncoef, const double* d_x,
                                  double* d_y, void* stream) {
  if (!h) return fail(B200MPC_ERR_ARG, "null handle");
  if (B < 0 || ncoef < 1 || ncoef > 64) return fail(B200MPC_ERR_ARG, "polyeval: bad B / ncoef");
  if (B == 0) return 0;
  if (!d_coeffs || !d_x || !d_y) return fail(B200MPC_ERR_ARG, "null pointer");
  CU(cudaSetDevice(h->device));
  CU(launch_polyeval(d_coeffs, ncoef, d_x, d_y, B, stream ? (cudaStream_t)stream : h->stream));
  h->launches += 1;
  return 0;
}

int b200mpc_polyeval_batch(b200mpc_handle* h, int B, const double* coeffs, int ncoef, const double* x, double* y) {
  if (!h) return fail(B200MPC_ERR_ARG, "null handle");
  if (B < 0 || ncoef < 1 || ncoef > 64) return fail(B200MPC_ERR_ARG, "polyeval: bad B / ncoef");
  if (B == 0) return 0;
  if (!coeffs || !x || !y) return fail(B200MPC_ERR_ARG, "null pointer");
  CU(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  const size_t nb = (size_t)B;
  CU(h->misc0.ensure(nb * (ncoef + 2) * sizeof(double)));   // coefficient rows | x | y
  double* a = h->misc0.as<double>();
  double* dy = a + nb * (ncoef + 1);
  CU(cudaMemcpyAsync(a, coeffs, nb * ncoef * sizeof(double), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(a + nb * ncoef, x, nb * sizeof(double), cudaMemcpyHostToDevice, s));
  CU(launch_polyeval(a, ncoef, a + nb * ncoef, dy, B, s, 1));
  h->launches += 1;
  CU(cudaMemcpyAsync(y, dy, nb * sizeof(double), cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  return 0;
}

int b200mpc_rollout_batch_device(b200mpc_handle* h, int B, int H, const double* d_state4, const double* d_act,
                                 double dt, double Lf, double* d_out, void* stream) {
  if (!h) return fail(B200MPC_ERR_ARG, "null handle");
  if (B < 0 || H < 1 || H > 4096) return fail(B200MPC_ERR_ARG, "rollout: bad B / H");
  if (!(Lf > 0)) return fail(B200MPC_ERR_ARG, "rollout: Lf must be positive");
  if (B == 0) return 0;
  if (!d_state4 || !d_act || !d_out) return fail(B200MPC_ERR_ARG, "null pointer");
  CU(cudaSetDevice(h->device));
  CU(launch_rollout(d_state4, d_act, B, H, dt, Lf, d_out, stream ? (cudaStream_t)stream : h->stream));
  h->launches += 1;
  return 0;
}

int b200mpc_rollout_batch(b200mpc_handle* h, int B, int H, const double* state4, const double* act, double dt,
                          double Lf, double* out) {
  if (!h) return fail(B200MPC_ERR_ARG, "null handle");
  if (B < 0 || H < 1 || H > 1024) return fail(B200MPC_ERR_ARG, "rollout: bad B / H (host entry: H <= 1024)");
  if (!(Lf > 0)) return fail(B200MPC_ERR_ARG, "rollout: Lf must be positive");
  if (B == 0) return 0;
  if (!state4 || !act || !out) return fail(B200MPC_ERR_ARG, "null pointer");
  CU(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  const size_t nb = (size_t)B, hh = (size_t)H;
  CU(h->misc0.ensure(nb * (4 + 2 * hh) * sizeof(double)));   // state rows | actuator rows
  CU(h->misc3.ensure(nb * 4 * hh * sizeof(double)));         // trajectory rows
  double* a = h->misc0.as<double>();
  CU(cudaMemcpyAsync(a, state4, nb * 4 * sizeof(double), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(a + nb * 4, act, nb * 2 * hh * sizeof(double), cudaMemcpyHostToDevice, s));
  CU(launch_rollout(a, a + nb * 4, B, H, dt, Lf, h->misc3.as<double>(), s, 1));
  h->launches += 1;
  CU(cudaMemcpyAsync(out, h->misc3.p, nb * 4 * hh * sizeof(double), cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  return 0;
}

int b200mpc_roadmap_reference_batch_device(b200mpc_handle* h, int B, const double* d_pose4, const double* d_centerline,
                                           int n_wp, double* d_state6_out, double* d_coeffs_out, void* stream) {
  if (!h) return fail(B200MPC_ERR_ARG, "null handle");
  if (B < 0 || n_wp < 6 || n_wp > 12000) return fail(B200MPC_ERR_ARG, "roadmap: need B >= 0 and 6 <= n_wp <= 12000");
  if (B == 0) return 0;
  if (!d_pose4 || !d_centerline || !d_state6_out || !d_coeffs_out) return fail(B200MPC_ERR_ARG, "null pointer");
  CU(cudaSetDevice(h->device));
  CU(launch_roadmap_reference(d_pose4, B, d_centerline, n_wp, d_state6_out, d_coeffs_out, stream ? (cudaStream_t)stream : h->stream));
  h->launches += 1;
  return 0;
}

int b200mpc_roadmap_reference_batch(b200mpc_handle* h, int B, const double* pose4, const double* centerline, int n_wp,
                                    double* state6_out, double* coeffs_out) {
  if (!h) return fail(B200MPC_ERR_ARG, "null handle");
  if (B < 0 || n_wp < 6 || n_wp > 12000) return fail(B200MPC_ERR_ARG, "roadmap: need B >= 0 and 6 <= n_wp <= 12000");
  if (B == 0) return 0;
  if (!pose4 || !centerline || !state6_out || !coeffs_out) return fail(B200MPC_ERR_ARG, "null pointer");
  CU(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  const size_t nb = (size_t)B;
  CU(h->misc0.ensure((nb * 4 + (size_t)2 * n_wp) * sizeof(double)));   // pose rows | centre line
  CU(h->misc3.ensure(nb * 10 * sizeof(double)));                        // state6 rows | coefficient rows
  double* a = h->misc0.as<double>();
  double* wp = a + nb * 4;
  double* ao = h->misc3.as<double>();
  CU(cudaMemcpyAsync(a, pose4, nb * 4 * sizeof(double), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(wp, centerline, (size_t)2 * n_wp * sizeof(double), cudaMemcpyHostToDevice, s));
  CU(launch_roadmap_reference(a, B, wp, n_wp, ao, ao + nb * 6, s, 1));
  h->launches += 1;
  CU(cudaMemcpyAsync(state6_out, ao, nb * 6 * sizeof(double), cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(coeffs_out, ao + nb * 6, nb * 4 * sizeof(double), cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  return 0;
}

// Host-side reader of the reference's roadmap file (no device work): one waypoint per line, fields split at ',' and
// converted one by one, as CustomMPC::parseRoadMapLine does (mpc_to_line/src/custom_MPC.h:35-44; std::stof there).
int b200mpc_read_roadmap_csv(const char* path, int float_fields, double* centerline_out, double* slope_out, int max_wp, int* n_wp) {
  if (!path || !n_wp) return fail(B200MPC_ERR_ARG, "null path / n_wp");
  if (max_wp < 0) return fail(B200MPC_ERR_ARG, "negative max_wp");
  std::ifstream f(path);
  if (!f.good()) return fail(B200MPC_ERR_ARG, std::string("cannot open roadmap file ") + path);
  std::string line;
  int n = 0, lineno = 0;
  while (std::getline(f, line)) {
    ++lineno;
    if (!line.empty() && line.back() == '\r') line.pop_back();
    if (line.find_first_not_of(" \t") == std::string::npos) continue;   // blank line
    std::istringstream ls(line);
    std::string number;
    double v[7];
    int k = 0;
    while (std::getline(ls, number, ',')) {
      if (k >= 7) { ++k; break; }
      try {
        size_t used = 0;
        v[k] = float_fields ? (double)std::stof(number, &used) : std::stod(number, &used);
      } catch (...) {
        return fail(B200MPC_ERR_ARG, std::string(path) + ":" + std::to_string(lineno) + ": field " + std::to_string(k + 1) + " is not a number");
      }
      ++k;
    }
    if (k != 7)
      return fail(B200MPC_ERR_ARG, std::string(path) + ":" + std::to_string(lineno) + ": expected 7 comma-separated fields (left x,y, right x,y, centre x,y, slope)");
    if (n < max_wp) {
      if (centerline_out) { centerline_out[2 * n] = v[4]; centerline_out[2 * n + 1] = v[5]; }
      if (slope_out) slope_out[n] = v[6];
    }
    ++n;
  }
  *n_wp = n;
  return 0;
}

// ------------------------------------------------------------------------------------------------
int b200mpc_set_timing(b200mpc_handle* h, int enable) {
  if (!h) return fail(B200MPC_ERR_ARG, "null handle");
  h->timing_on = enable != 0;
  return 0;
}

int b200mpc_kernel_time_ms(b200mpc_handle* h, double* total_ms, int* launches, int reset) {
  if (!h) return fail(B200MPC_ERR_ARG, "null handle");
  CU(cudaSetDevice(h->device));
  double tot = 0.0;
  for (auto& ev : h->timing) {
    CU(cudaEventSynchronize(ev.second));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, ev.first, ev.second));
    tot += ms;
  }
  if (total_ms) *total_ms = tot;
  if (launches) *launches = (int)h->timing.size();
  if (reset) {
    for (auto& ev : h->timing) { cudaEventDestroy(ev.first); cudaEventDestroy(ev.second); }
    h->timing.clear();
  }
  return 0;
}

int b200mpc_selftest_division(b200mpc_handle* h, int n, const double* a, const double* b, double* quot, double* rcp) {
  if (!h) return fail(B200MPC_ERR_ARG, "null handle");
  if (n < 0) return fail(B200MPC_ERR_ARG, "negative count");
  if (n == 0) return 0;
  if (!a || !b || !quot || !rcp) return fail(B200MPC_ERR_ARG, "null operand / result array");
  CU(cudaSetDevice(h->device));
  const size_t bytes = (size_t)n * sizeof(double);
  CU(h->misc3.ensure(4 * bytes));
  double* d = h->misc3.as<double>();
  cudaStream_t s = h->stream;
  CU(cudaMemcpyAsync(d, a, bytes, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(d + n, b, bytes, cudaMemcpyHostToDevice, s));
  CU(launch_division_selftest(n, d, d + n, d + 2 * (size_t)n, d + 3 * (size_t)n, s));
  CU(cudaMemcpyAsync(quot, d + 2 * (size_t)n, bytes, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(rcp, d + 3 * (size_t)n, bytes, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  h->launches += 1;
  return 0;
}

int b200mpc_measure_fp64_peak(b200mpc_handle* h, double* tflops) {
  if (!h || !tflops) return fail(B200MPC_ERR_ARG, "null handle / output");
  CU(cudaSetDevice(h->device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, h->device));
  CU(h->misc0.ensure(1024));
  cudaStream_t s = h->stream;
  cudaEvent_t e0, e1;
  CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
  const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
  double flop = 0.0, best = 0.0;
  CU(launch_fp64_peak(h->misc0.as<double>(), blocks, threads, 64, s, &flop));   // warm-up
  for (int rep = 0; rep < 5; ++rep) {
    CU(cudaEventRecord(e0, s));
    CU(launch_fp64_peak(h->misc0.as<double>(), blocks, threads, iters, s, &flop));
    CU(cudaEventRecord(e1, s));
    CU(cudaEventSynchronize(e1));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, e0, e1));
    const double tf = flop / (ms * 1e-3) / 1e12;
    if (tf > best) best = tf;
  }
  h->launches += 6;
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  *tflops = best;
  return 0;
}

}  // extern "C"
