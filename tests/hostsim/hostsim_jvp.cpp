// TEST INFRASTRUCTURE ONLY: the solver core's forward sensitivities (udacitympc_b200/csrc/mpc_core.cuh, Solver::jvp<true>,
// the arithmetic of the per-problem-model JVP instance) compiled for the CPU, so the JVP can be checked against the VJP,
// a dense KKT solve and finite differences without a GPU.  Built next to hostsim_sens_model.cpp as libhostsim_jvp.so;
// NOT part of libb200mpc.so.
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
    std::fprintf(stderr, "hostsim_jvp: workspace index %d out of range [0, %d)\n", i, g_ws_limit);
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

// The JVP of one problem at (traj (8N-2), mult (10N-4)) along (t_state6 (6), t_coeffs (ncoef), t_cost8 (8), t_model4 (4));
// any tangent may be null (zero).  Writes t_out8 (8), t_traj (8N-2), *t_obj; returns the status of b200mpc_solve_batch_jvp.
int hostsim_jvp(const hostsim_params* hp, const double* state6, const double* coeffs, int ncoef, const double* traj,
                const double* mult, const double* t_state6, const double* t_coeffs, const double* t_cost8,
                const double* t_model4, double* t_out8, double* t_traj, double* t_obj) {
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
  double ts6[6], tcf[kMaxCoef], tpar[8], tmod[4];
  for (int k = 0; k < 6; ++k) ts6[k] = t_state6 ? t_state6[k] : 0.0;
  for (int i = 0; i < kMaxCoef; ++i) tcf[i] = t_coeffs && i < ncoef ? t_coeffs[i] : 0.0;
  for (int i = 0; i < 8; ++i) tpar[i] = t_cost8 ? t_cost8[i] : 0.0;
  for (int i = 0; i < 4; ++i) tmod[i] = t_model4 ? t_model4[i] : 0.0;
  return S.jvp<true>(state6, traj, 1, mult, 1, ts6, tcf, tpar, tmod, t_traj, 1, t_out8, 1, *t_obj);
}
}
