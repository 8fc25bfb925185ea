// TEST INFRASTRUCTURE ONLY: compiles the solver core (udacitympc_b200/csrc/mpc_core.cuh) for the CPU so the
// algorithm can be checked against the oracle in the GPU-less build container (pytest -m "not gpu").
// It is NOT part of libb200mpc.so and is never used by the product path.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <vector>

#define MPC_BOUNDS_CHECK 1
#include "../../udacitympc_b200/csrc/mpc_core.cuh"
#include "../../udacitympc_b200/csrc/mpc_coop.cuh"

// every workspace access of the solver core is range-checked in this build
static thread_local int g_ws_limit = 0;
namespace b200mpc {
void mpc_bounds_check(int i) {
  if (i < 0 || i >= g_ws_limit) {
    std::fprintf(stderr, "hostsim: workspace index %d out of range [0, %d)\n", i, g_ws_limit);
    std::abort();
  }
}
}  // namespace b200mpc

using namespace b200mpc;

struct HostExec {   // the cooperative solver's primitives on one CPU thread: lanes run one after the other
  bool lane0() const { return true; }
  void sync() const {}
  template <class F>
  void for_stages(int n, F f) const {
    for (int t = 0; t < n; ++t) f(t);
  }
};

extern "C" {
struct hostsim_params {
  int N;
  double dt, Lf, ref_v, w_cte, w_epsi, w_v, w_delta, w_a, w_ddelta, w_da, delta_max, a_max, tol;
  int max_iter;
};
static int g_resto = 2;   // Params::resto of the following solves (0 off, 1 restoration step, 2 soft restoration phase first)
void hostsim_set_restoration(int mode) { g_resto = mode; }


// trace rows of 8: iter, mu, alpha_pr, alpha_du, dw, f, theta, phase-trips
// mode 0: one Solver object loops trip() (what the single fused kernel does)
// mode 1: every pass runs on a FRESH Solver object whose scalar state is loaded from / stored to the workspace
//         (what the per-pass kernels do) -- catches any state that is not persisted.
int hostsim_solve_mode(const hostsim_params* hp, const double* state6, const double* coeffs, int ncoef, double* x_out,
                       double* out8, double* obj, int* iters, double* lam_out, double* trace, int trace_cap,
                       int* trace_rows, int mode) {
  Params P;
  P.N = hp->N; P.dt = hp->dt; P.Lf = hp->Lf; P.ref_v = hp->ref_v;
  P.w_cte = hp->w_cte; P.w_epsi = hp->w_epsi; P.w_v = hp->w_v; P.w_delta = hp->w_delta; P.w_a = hp->w_a;
  P.w_ddelta = hp->w_ddelta; P.w_da = hp->w_da; P.delta_max = hp->delta_max; P.a_max = hp->a_max; P.tol = hp->tol;
  P.max_iter = hp->max_iter;
  P.resto = g_resto;
  P.finalize();
  std::vector<double> ws((size_t)workspace_doubles_per_problem(P.N), 0.0);
  g_ws_limit = (int)ws.size();
  int rows = 0, trips = 0, last_iter = -1;
  Result R;
  double df = 1.0;
  int cur = 0;
  auto log_row = [&](Solver<1>& S) {
    if (trace && S.iter != last_iter && rows < trace_cap) {
      double* r = trace + 8 * rows++;
      r[0] = S.iter; r[1] = S.mu; r[2] = S.alpha; r[3] = S.alpha_du; r[4] = S.dw_curr; r[5] = S.f_cur / S.df;
      r[6] = S.theta_cur; r[7] = trips;
      last_iter = S.iter;
    }
  };
  if (mode >= 2) {
    // cooperative (warp-per-problem) solver.  mode 2: from the start.  mode 3+: the thread version runs the first
    // (mode - 3) trips / passes, then the cooperative solver takes the problem over wherever it is.
    Solver<1> S(P, ws.data());
    double carry[kCarry];
    S.cr = carry; S.cs = 1;
    std::vector<CoopStage> st((size_t)P.N);
    CoopPub pub;
    CoopSolver<1, HostExec> C(S, st.data(), &pub, HostExec{});
    if (mode == 2) { S.set_coeffs(coeffs, ncoef); C.init(state6); }
    else S.init(state6, coeffs, ncoef);
    if (mode >= 3) {
      int passes = mode - 3;
      while (S.phase != PH_DONE && passes > 0) {   // one pass at a time so the hand-over can happen in any phase
        if (S.phase == PH_FACTOR) S.do_factor();
        else if (S.phase == PH_FORWARD) S.do_forward();
        else S.do_step();
        --passes;
      }
    }
    C.run();
    S.finish(R, x_out, 1);
    df = S.df; cur = S.cur;
    trips = S.iter;
  } else if (mode == 0) {
    Solver<1> S(P, ws.data());
    double carry[kCarry];
    S.cr = carry; S.cs = 1;
    S.init(state6, coeffs, ncoef);
    while (S.phase != PH_DONE && trips < 100000) { S.trip(); ++trips; log_row(S); }
    S.finish(R, x_out, 1);
    df = S.df; cur = S.cur;
  } else {
    // mode -1 / -2: as mode 1, and the problem is moved to another workspace (repack_problem, what the batch
    // compaction does) after every round / after every pass; the destination is poisoned with NaN first, so anything
    // the move leaves behind that a later pass reads shows up in the results.
    { Solver<1> S(P, ws.data()); S.init(state6, coeffs, ncoef); S.store_state(); }
    std::vector<double> other(ws.size());
    auto repack = [&]() {
      for (auto& v : other) v = std::nan("");
      repack_problem(P, Ws<1>{ws.data(), 0}, Ws<1>{other.data(), 0});
      ws.swap(other);
    };
    int phase = PH_FACTOR;
    while (phase != PH_DONE && trips < 400000) {
      for (int k = 0; k < 3; ++k) {   // the three kernels of one round
        Solver<1> S(P, ws.data());
        double carry[kCarry];
        S.cr = carry; S.cs = 1;
        if (S.load_phase() != k) continue;
        S.set_coeffs(coeffs, ncoef);
        if (k == PH_FACTOR) S.kernel_factor();
        else if (k == PH_FORWARD) S.kernel_forward();
        else S.kernel_step();
        phase = S.load_phase();
        if (k == PH_STEP) { S.load_state(); log_row(S); }
        if (mode == -2 && phase != PH_DONE) repack();
      }
      if (phase == PH_RESTO) {   // the per-pass kernels leave it to the finisher, which runs the problem to completion
        Solver<1> S(P, ws.data());
        double carry[kCarry];
        S.cr = carry; S.cs = 1;
        S.set_coeffs(coeffs, ncoef);
        S.load_state();
        while (S.phase != PH_DONE && trips < 400000) { S.trip(); ++trips; log_row(S); }
        S.store_state();
        phase = S.load_phase();
      }
      if (mode == -1 && phase != PH_DONE) repack();
      ++trips;
    }
    Solver<1> S(P, ws.data());
    S.set_coeffs(coeffs, ncoef);
    S.load_state();
    S.finish(R, x_out, 1);
    df = S.df; cur = S.cur;
  }
  for (int i = 0; i < 8; ++i) out8[i] = R.out8[i];
  *obj = R.obj; *iters = R.iters;
  if (lam_out) for (int t = 0; t < P.N; ++t) for (int k = 0; k < 6; ++k) lam_out[k * P.N + t] = ws[(size_t)(t + 1) * kRec + kX * cur + xLAM + k] / df;
  if (trace_rows) *trace_rows = rows;
  return R.status;
}

// closed loop of solution/main.cpp:51-76 on one Solver object: `steps` solves, each fed the previous solve's predicted
// state; warm != 0: steps after the first start from the shifted previous solution (Solver::init_warm)
int hostsim_closed_loop(const hostsim_params* hp, const double* state6, const double* coeffs, int ncoef, int steps, int warm,
                        double mu0, double* hist8, int* iters, int* status) {
  Params P;
  P.N = hp->N; P.dt = hp->dt; P.Lf = hp->Lf; P.ref_v = hp->ref_v;
  P.w_cte = hp->w_cte; P.w_epsi = hp->w_epsi; P.w_v = hp->w_v; P.w_delta = hp->w_delta; P.w_a = hp->w_a;
  P.w_ddelta = hp->w_ddelta; P.w_da = hp->w_da; P.delta_max = hp->delta_max; P.a_max = hp->a_max; P.tol = hp->tol;
  P.max_iter = hp->max_iter;
  P.resto = g_resto;
  P.finalize();
  std::vector<double> ws((size_t)workspace_doubles_per_problem(P.N), 0.0);
  g_ws_limit = (int)ws.size();
  double s0[6];
  for (int k = 0; k < 6; ++k) s0[k] = state6[k];
  for (int step = 0; step < steps; ++step) {
    Solver<1> S(P, ws.data());
    double carry[kCarry];
    S.cr = carry; S.cs = 1;
    S.set_coeffs(coeffs, ncoef);
    if (warm && step > 0) S.init_warm(s0, mu0);
    else S.init(s0, coeffs, ncoef);
    int trips = 0;
    while (S.phase != PH_DONE && trips < 100000) { S.trip(); ++trips; }
    S.store_state();
    Result R;
    S.finish(R, nullptr, 1);
    for (int k = 0; k < 8; ++k) hist8[8 * step + k] = R.out8[k];
    iters[step] = R.iters; status[step] = R.status;
    for (int k = 0; k < 6; ++k) s0[k] = R.out8[k];
  }
  return 0;
}

// The DEVICE memory layout on the host: B problems in warp-interleaved groups of 32 (Solver<32>, element i of slot s at
// region[((s >> 5) * doubles_per_problem + i) * 32 + (s & 31)], the arithmetic of slot_base() / region_doubles() in
// solve_kernel.cu), two regions, per-pass execution with the scalar state reloaded for every pass, and after every
// round (compact != 0) the batch compaction: the live problems move to consecutive slots of the other region, which is
// poisoned with NaN first.  Guard words behind both regions catch any write outside a region.  Returns 0, or -1 if a
// guard word changed.
// max_rounds > 0: after that many rounds the finisher takes every live problem over (coop != 0: the cooperative solver,
// else the thread-per-problem loop), as launch_solve does on the device.
int hostsim_batch_interleaved(const hostsim_params* hp, int B, const double* states, const double* coeffs, int ncoef,
                              int compact, int max_rounds, int coop, double* out8, double* obj, int* iters, int* status) {
  Params P;
  P.N = hp->N; P.dt = hp->dt; P.Lf = hp->Lf; P.ref_v = hp->ref_v;
  P.w_cte = hp->w_cte; P.w_epsi = hp->w_epsi; P.w_v = hp->w_v; P.w_delta = hp->w_delta; P.w_a = hp->w_a;
  P.w_ddelta = hp->w_ddelta; P.w_da = hp->w_da; P.delta_max = hp->delta_max; P.a_max = hp->a_max; P.tol = hp->tol;
  P.max_iter = hp->max_iter;
  P.resto = g_resto;
  P.finalize();
  const size_t wdpp = (size_t)workspace_doubles_per_problem(P.N), groups = ((size_t)B + 31) / 32, region = groups * wdpp * 32;
  const size_t guard = 4096;
  const double kGuard = -7.25e77;
  std::vector<double> mem[2];
  for (auto& m : mem) { m.assign(region + guard, std::nan("")); for (size_t i = region; i < region + guard; ++i) m[i] = kGuard; }
  g_ws_limit = (int)wdpp;
  auto base = [&](int r, int slot) { return mem[r].data() + (size_t)(slot >> 5) * wdpp * 32 + (slot & 31); };
  std::vector<int> prob(B), where(B);   // slot -> problem of the current region, problem -> slot
  for (int b = 0; b < B; ++b) { prob[b] = b; where[b] = b; }
  int cur = 0, occupied = B;
  for (int b = 0; b < B; ++b) {
    Solver<32> S(P, base(0, b), b & 31);
    S.init(states + 6 * b, coeffs + (size_t)ncoef * b, ncoef);
    S.store_state();
  }
  std::vector<char> done(B, 0);
  auto finish = [&](int slot) {
    const int b = prob[slot];
    Solver<32> S(P, base(cur, slot), slot & 31);
    S.set_coeffs(coeffs + (size_t)ncoef * b, ncoef);
    S.load_state();
    Result R;
    S.finish(R, nullptr, 1);
    for (int k = 0; k < 8; ++k) out8[8 * b + k] = R.out8[k];
    obj[b] = R.obj; iters[b] = R.iters; status[b] = R.status;
    done[b] = 1;
  };
  for (int round = 0; round < 100000; ++round) {
    int live = 0;
    for (int slot = 0; slot < occupied; ++slot) {
      const int b = prob[slot];
      if (done[b]) continue;
      for (int k = 0; k < 3; ++k) {
        Solver<32> S(P, base(cur, slot), slot & 31);
        double carry[kCarry];
        S.cr = carry; S.cs = 1;
        if (S.load_phase() != k) continue;
        S.set_coeffs(coeffs + (size_t)ncoef * b, ncoef);
        if (k == PH_FACTOR) S.kernel_factor();
        else if (k == PH_FORWARD) S.kernel_forward();
        else S.kernel_step();
      }
      Solver<32> S(P, base(cur, slot), slot & 31);
      if (S.load_phase() == PH_RESTO || (max_rounds > 0 && round + 1 >= max_rounds && S.load_phase() != PH_DONE)) {   // finisher
        double carry[kCarry];
        S.cr = carry; S.cs = 1;
        S.set_coeffs(coeffs + (size_t)ncoef * b, ncoef);
        S.load_state();
        if (coop) {
          std::vector<CoopStage> stg((size_t)P.N);
          CoopPub pub;
          CoopSolver<32, HostExec> C(S, stg.data(), &pub, HostExec{});
          C.run();
        } else {
          int guard_trips = 0;
          while (S.phase != PH_DONE && guard_trips++ < 400000) S.trip();
        }
        S.store_state();
      }
      if (S.load_phase() == PH_DONE) finish(slot);
      else ++live;
    }
    if (live == 0) break;
    if (compact) {   // live problems to consecutive slots of the other region, in reverse order for good measure
      const int other = cur ^ 1;
      for (size_t i = 0; i < region; ++i) mem[other][i] = std::nan("");
      std::vector<int> np_;
      for (int slot = occupied - 1; slot >= 0; --slot) {
        const int b = prob[slot];
        if (done[b]) continue;
        const int ds = (int)np_.size();
        repack_problem(P, Ws<32>{base(cur, slot), slot & 31}, Ws<32>{base(other, ds), ds & 31});
        np_.push_back(b);
      }
      for (size_t i = 0; i < np_.size(); ++i) { prob[i] = np_[i]; where[np_[i]] = (int)i; }
      occupied = (int)np_.size();
      cur = other;
    }
  }
  for (auto& m : mem)
    for (size_t i = region; i < region + guard; ++i)
      if (m[i] != kGuard) return -1;
  return 0;
}

int hostsim_solve(const hostsim_params* hp, const double* state6, const double* coeffs, int ncoef, double* x_out,
                  double* out8, double* obj, int* iters, double* lam_out, double* trace, int trace_cap, int* trace_rows) {
  return hostsim_solve_mode(hp, state6, coeffs, ncoef, x_out, out8, obj, iters, lam_out, trace, trace_cap, trace_rows, 0);
}
}
