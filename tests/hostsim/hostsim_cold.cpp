// TEST INFRASTRUCTURE ONLY: the solver core (udacitympc_b200/csrc/mpc_core.cuh) compiled for the CPU to check the cold
// start of the init kernel (Solver::kernel_ls_round: the multiplier-initialisation round on the start point in closed
// form) against the per-pass round it replaces, bit for bit.  Built next to hostsim.cpp as libhostsim_cold.so; NOT part of
// libb200mpc.so.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <vector>

#define MPC_BOUNDS_CHECK 1
#include "../../udacitympc_b200/csrc/mpc_core.cuh"

// every workspace access of the solver core is range-checked in this build
static thread_local int g_ws_limit = 0;
namespace b200mpc {
void mpc_bounds_check(int i) {
  if (i < 0 || i >= g_ws_limit) {
    std::fprintf(stderr, "hostsim_cold: workspace index %d out of range [0, %d)\n", i, g_ws_limit);
    std::abort();
  }
}
}  // namespace b200mpc

using namespace b200mpc;

namespace {
// one pass of the per-pass kernels on the problem in ws (phase: its phase), or the finisher for PH_RESTO
void pass(const Params& P, double* ws, const double* coeffs, int ncoef, int phase) {
  Solver<1> S(P, ws);
  double carry[kCarry];
  S.cr = carry; S.cs = 1;
  S.set_coeffs(coeffs, ncoef);
  if (phase == PH_FACTOR) S.kernel_factor();
  else if (phase == PH_FORWARD) S.kernel_forward();
  else if (phase == PH_STEP) S.kernel_step();
  else {
    S.load_state();
    while (S.phase != PH_DONE) S.trip();
    S.store_state();
  }
}
}  // namespace

extern "C" {
struct hostsim_params {   // same layout as tests/hostsim/hostsim.cpp and oracle_bindings.OracleParams
  int N;
  double dt, Lf, ref_v, w_cte, w_epsi, w_v, w_delta, w_a, w_ddelta, w_da, delta_max, a_max, tol;
  int max_iter;
};

// One cold solve, two ways, each in a NaN-poisoned workspace of workspace_doubles_per_problem(N) doubles:
//   path 0 (the per-pass round): init, then the factor / forward / step passes of the per-pass kernels until the
//          multiplier-initialisation round is over (F_LS cleared) or the problem is finished;
//   path 1 (the init kernel): init, then Solver::kernel_ls_round.
// ws_after[2][n]: both workspaces at that point.  Then both run the per-pass passes to the end: out8[2][8], obj[2],
// iters[2], status[2], x_out[2][8N-2].  *kept: the estimate was kept (F_LSKEEP seen on path 0).  Returns 0, or -1 if
// path 0 did not leave the round within 8 passes.
int hostsim_cold_compare(const hostsim_params* hp, const double* state6, const double* coeffs, int ncoef, double* ws_after,
                         double* out8, double* obj, int* iters, int* status, double* x_out, int* kept) {
  Params P;
  P.N = hp->N; P.dt = hp->dt; P.Lf = hp->Lf; P.ref_v = hp->ref_v;
  P.w_cte = hp->w_cte; P.w_epsi = hp->w_epsi; P.w_v = hp->w_v; P.w_delta = hp->w_delta; P.w_a = hp->w_a;
  P.w_ddelta = hp->w_ddelta; P.w_da = hp->w_da; P.delta_max = hp->delta_max; P.a_max = hp->a_max; P.tol = hp->tol;
  P.max_iter = hp->max_iter;
  P.resto = 2;   // the library default (soft restoration phase, then the restoration step)
  P.finalize();
  const size_t n = (size_t)workspace_doubles_per_problem(P.N);
  g_ws_limit = (int)n;
  *kept = 0;
  for (int path = 0; path < 2; ++path) {
    std::vector<double> ws(n, std::nan(""));
    {
      Solver<1> S(P, ws.data());
      S.init(state6, coeffs, ncoef);
      S.store_state();
      if (path == 1 && S.phase == PH_FACTOR) S.kernel_ls_round(state6);
    }
    int phase = Solver<1>(P, ws.data()).load_phase();
    if (path == 0) {
      int passes = 0;
      while (((int)ws[iFLAGS] & F_LS) && phase != PH_DONE) {
        if (++passes > 8) return -1;
        pass(P, ws.data(), coeffs, ncoef, phase);
        if ((int)ws[iFLAGS] & F_LSKEEP) *kept = 1;
        phase = Solver<1>(P, ws.data()).load_phase();
      }
    }
    for (size_t i = 0; i < n; ++i) ws_after[path * n + i] = ws[i];
    for (int trips = 0; phase != PH_DONE && trips < 400000; ++trips) {
      pass(P, ws.data(), coeffs, ncoef, phase);
      phase = Solver<1>(P, ws.data()).load_phase();
    }
    Solver<1> S(P, ws.data());
    S.set_coeffs(coeffs, ncoef);
    S.load_state();
    Result R;
    S.finish(R, x_out + (size_t)path * (8 * P.N - 2), 1);
    for (int k = 0; k < 8; ++k) out8[8 * path + k] = R.out8[k];
    obj[path] = R.obj; iters[path] = R.iters; status[path] = R.status;
  }
  return 0;
}
}
