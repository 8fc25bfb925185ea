// TEST INFRASTRUCTURE ONLY: the solver core (udacitympc_b200/csrc/mpc_core.cuh, mpc_coop.cuh) compiled for the CPU to
// check the warm start from a caller-supplied point (Solver::init_guess, CoopSolver::init_guess) and the multiplier
// output (Solver::finish) without a GPU.  Built next to hostsim.cpp as libhostsim_guess.so; NOT part of libb200mpc.so.
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
    std::fprintf(stderr, "hostsim_guess: workspace index %d out of range [0, %d)\n", i, g_ws_limit);
    std::abort();
  }
}
}  // namespace b200mpc

using namespace b200mpc;

namespace {
struct HostExec {   // the cooperative solver's primitives on one CPU thread: lanes run one after the other
  bool lane0() const { return true; }
  void sync() const {}
  template <class F>
  void for_stages(int n, F f) const {
    for (int t = 0; t < n; ++t) f(t);
  }
};
}  // namespace

extern "C" {
struct hostsim_params {   // same layout as tests/hostsim/hostsim.cpp and oracle_bindings.OracleParams
  int N;
  double dt, Lf, ref_v, w_cte, w_epsi, w_v, w_delta, w_a, w_ddelta, w_da, delta_max, a_max, tol;
  int max_iter;
};

// One solve from a caller-supplied primal-dual point (x_init == null: the default start point; mult_init may be null),
// returning the solution x_out (8N-2), out8, obj, iters and the multipliers mult_out (10N-4, layout of Solver::finish).
// mode 0: one Solver object loops trip() (the fused kernel); -2: every pass on a fresh Solver object whose scalar state is
// loaded from / stored to the workspace (the per-pass kernels), the problem moved to a NaN-poisoned workspace after every
// pass (the batch compaction); 2: the cooperative solver from the start (the cooperative kernel).
int hostsim_solve_guess(const hostsim_params* hp, const double* state6, const double* coeffs, int ncoef, const double* x_init,
                        const double* mult_init, double mu_init, double* x_out, double* out8, double* obj, int* iters,
                        double* mult_out, int mode) {
  Params P;
  P.N = hp->N; P.dt = hp->dt; P.Lf = hp->Lf; P.ref_v = hp->ref_v;
  P.w_cte = hp->w_cte; P.w_epsi = hp->w_epsi; P.w_v = hp->w_v; P.w_delta = hp->w_delta; P.w_a = hp->w_a;
  P.w_ddelta = hp->w_ddelta; P.w_da = hp->w_da; P.delta_max = hp->delta_max; P.a_max = hp->a_max; P.tol = hp->tol;
  P.max_iter = hp->max_iter;
  P.resto = 2;   // the library default (soft restoration phase, then the restoration step)
  P.finalize();
  std::vector<double> ws((size_t)workspace_doubles_per_problem(P.N), 0.0);
  g_ws_limit = (int)ws.size();
  auto start = [&](Solver<1>& S) {
    S.set_coeffs(coeffs, ncoef);
    if (x_init) S.init_guess(state6, x_init, 1, mult_init, 1, mu_init);
    else S.init(state6, coeffs, ncoef);
  };
  Result R;
  if (mode == 2) {
    Solver<1> S(P, ws.data());
    double carry[kCarry];
    S.cr = carry; S.cs = 1;
    std::vector<CoopStage> st((size_t)P.N);
    CoopPub pub;
    CoopSolver<1, HostExec> C(S, st.data(), &pub, HostExec{});
    S.set_coeffs(coeffs, ncoef);
    if (x_init) C.init_guess(state6, x_init, 1, mult_init, 1, mu_init);
    else C.init(state6);
    C.run();
    S.finish(R, x_out, 1, mult_out);
  } else if (mode == 0) {
    Solver<1> S(P, ws.data());
    double carry[kCarry];
    S.cr = carry; S.cs = 1;
    start(S);
    for (int trips = 0; S.phase != PH_DONE && trips < 100000; ++trips) S.trip();
    S.finish(R, x_out, 1, mult_out);
  } else if (mode == -2) {
    { Solver<1> S(P, ws.data()); start(S); S.store_state(); }
    std::vector<double> other(ws.size());
    int phase = Solver<1>(P, ws.data()).load_phase();
    for (int trips = 0; phase != PH_DONE && trips < 400000; ++trips) {
      Solver<1> S(P, ws.data());
      double carry[kCarry];
      S.cr = carry; S.cs = 1;
      S.set_coeffs(coeffs, ncoef);
      if (phase == PH_FACTOR) S.kernel_factor();
      else if (phase == PH_FORWARD) S.kernel_forward();
      else if (phase == PH_STEP) S.kernel_step();
      else {   // PH_RESTO: the per-pass kernels leave it to the finisher, which runs the problem to completion
        S.load_state();
        while (S.phase != PH_DONE) S.trip();
        S.store_state();
      }
      phase = S.load_phase();
      if (phase != PH_DONE) {
        for (auto& v : other) v = std::nan("");
        repack_problem(P, Ws<1>{ws.data(), 0}, Ws<1>{other.data(), 0});
        ws.swap(other);
      }
    }
    Solver<1> S(P, ws.data());
    S.set_coeffs(coeffs, ncoef);
    S.load_state();
    S.finish(R, x_out, 1, mult_out);
  } else {
    return -1000;
  }
  for (int i = 0; i < 8; ++i) out8[i] = R.out8[i];
  *obj = R.obj; *iters = R.iters;
  return R.status;
}
}
