// TEST INFRASTRUCTURE ONLY: the solver core's adjoint sensitivities with the vehicle-model gradient
// (udacitympc_b200/csrc/mpc_core.cuh, Solver::vjp<true>, the arithmetic of the per-problem-model VJP instance) compiled for
// the CPU, so grad_model can be checked against a dense KKT solve without a GPU.  Built next to hostsim_sens.cpp as
// libhostsim_sens_model.so; NOT part of libb200mpc.so.
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
    std::fprintf(stderr, "hostsim_sens_model: workspace index %d out of range [0, %d)\n", i, g_ws_limit);
    std::abort();
  }
}
}  // namespace b200mpc

using namespace b200mpc;

extern "C" {
struct hostsim_params {   // same layout as tests/hostsim/hostsim.cpp and oracle_bindings.OracleParams
  int N;
  double dt, Lf, ref_v, w_cte, w_epsi, w_v, w_delta, w_a, w_ddelta, w_da, delta_max, a_max, tol;
  int max_iter;
};

// The VJP of one problem at (traj (8N-2), mult (10N-4)) as hostsim_vjp (hostsim_sens.cpp) returns it, plus grad_model
// (4: dt, Lf, delta_max, a_max).  Returns the status of b200mpc_solve_batch_vjp_model.
int hostsim_vjp_model(const hostsim_params* hp, const double* state6, const double* coeffs, int ncoef, const double* traj,
                      const double* mult, const double* g_out8, const double* g_traj, double g_obj, double* grad_state6,
                      double* grad_coeffs, double* grad_params, double* grad_model) {
  Params P;
  P.N = hp->N; P.dt = hp->dt; P.Lf = hp->Lf; P.ref_v = hp->ref_v;
  P.w_cte = hp->w_cte; P.w_epsi = hp->w_epsi; P.w_v = hp->w_v; P.w_delta = hp->w_delta; P.w_a = hp->w_a;
  P.w_ddelta = hp->w_ddelta; P.w_da = hp->w_da; P.delta_max = hp->delta_max; P.a_max = hp->a_max; P.tol = hp->tol;
  P.max_iter = hp->max_iter;
  P.resto = 2;
  P.finalize();
  std::vector<double> ws((size_t)workspace_doubles_per_problem(P.N), std::nan(""));
  g_ws_limit = (int)ws.size();
  Solver<1> S(P, ws.data());
  S.set_coeffs(coeffs, ncoef);
  double gcf[kMaxCoef];
  const int st = S.vjp<true>(state6, traj, 1, mult, 1, g_out8, 1, g_traj, 1, g_obj, grad_state6, gcf, grad_params, grad_model);
  for (int i = 0; i < ncoef; ++i) grad_coeffs[i] = gcf[i];
  return st;
}
}
