// Launchers of the sm_100a kernels behind the C ABI (include/b200mpc.h).  Device pointers only.
#pragma once
#include <cuda_runtime.h>

#include "mpc_core.cuh"

namespace b200mpc {

// doubles of workspace needed to solve B problems at horizon N
size_t solve_workspace_doubles(int N, int B);

// call once per device before the first solve on it
cudaError_t solver_prepare_device();

enum SolveMode { kModePerPass = 0, kModeFused = 1 };
struct SolveConfig {
  int mode = kModePerPass;
  // per-pass mode: rounds of (factor, forward, step) before the finisher takes the thin tail.  0 = automatic: adaptive
  // hand-over (below); without batch compaction 18, or 16 when the call is cut into concurrent sub-batches
  int rounds = 0;
  int fused_below = 3072; // batches smaller than this skip the per-pass rounds (one launch: latency path)
  bool warm_start = false;   // closed loop only: steps after the first start from the shifted previous solution
  double warm_mu = 1e-4;     // barrier parameter a warm-started solve begins with
  int split = 4;             // large batches run as this many concurrent parts (see launch_solve)
  // adaptive hand-over (automatic rounds only): occupied slots (whole call) at which the cooperative kernel takes over
  int handover_below = 1184;      // one wave of 8 warps on 148 SMs
  int handover_from = 14;         // first round after which it may happen
  // batch compaction: after every round from compact_from on, if the unfinished problems fill at most
  // compact_max_live of the occupied workspace slots, they are moved to consecutive slots, so that later rounds run
  // full warps on whole 32-byte sectors (0 = off)
  double compact_max_live = 0.7;
  int compact_from = 4;
  bool coop = true;       // latency path = cooperative warp-per-problem kernel (false: thread-per-problem fused kernel)
};
struct SplitStreams {   // auxiliary streams / events owned by the handle (n_aux <= 3)
  int n_aux = 0;
  cudaStream_t aux[3] = {nullptr, nullptr, nullptr};
  cudaEvent_t fork = nullptr, join[3] = {nullptr, nullptr, nullptr};
};
// The per-call buffers of a solve (device pointers).  io_aos = 0: field-major (SoA) over the batch
//   state6 [6][B], coeffs [ncoef][B], out8 [steps][8][B], traj [8N-2][B] (last step, optional),
//   obj [steps][B] (optional), status [B] (last step, optional), iters [steps][B] (optional),
//   x_init [8N-2][B] + mult_init [10N-4][B] (optional: start from this point with barrier parameter mu_init instead of
//   the default start point, Solver::init_guess; mult_init may be null), mult [10N-4][B] (last step, optional),
//   cost8 [8][B] (optional: per-problem ref_v, w_cte, w_epsi, w_v, w_delta, w_a, w_ddelta, w_da instead of the handle's),
//   model4 [4][B] (optional: per-problem dt, Lf, delta_max, a_max instead of the handle's);
// io_aos = 1: state6 [B][6], coeffs [B][ncoef], out8 [steps][B][8] (reference order), cost8 [B][8], model4 [B][4], the
// others as above
struct SolveIO {
  const double *state6 = nullptr, *coeffs = nullptr;
  int ncoef = 0;
  double *out8 = nullptr, *traj = nullptr, *obj = nullptr;
  int *status = nullptr, *iters = nullptr;
  int io_aos = 0;
  const double *x_init = nullptr, *mult_init = nullptr;
  double mu_init = 0.0;
  double* mult = nullptr;
  const double* cost8 = nullptr;
  const double* model4 = nullptr;
};

// K1+K2+K3 fused: `steps` consecutive interior-point solves per problem (steps > 1 = closed loop, each solve
// starting from the previous solve's predicted state).  The launchers add one to *n_launches per kernel they launch.
cudaError_t launch_solve(const Params& P, int B, int steps, const SolveIO& io, double* ws, const SolveConfig& cfg,
                         cudaStream_t stream, const SplitStreams* ss, long long* n_launches);

// Pipelined solves: one solve (steps = 1) as two launch sequences (see solve_kernel.cu).  A tail context is a workspace
// of solve_workspace_doubles(N, slots) doubles.
struct TailCtx {
  double* ws = nullptr;
  int slots = 0;
};
cudaError_t launch_solve_bulk(const Params& P, int B, const SolveIO& io, double* ws, const TailCtx& tail, const SolveConfig& cfg,
                              cudaStream_t stream, long long* n_launches);
cudaError_t launch_solve_tail(const Params& P, int B, const SolveIO& io, const TailCtx& tail, const SolveConfig& cfg,
                              cudaStream_t stream, long long* n_launches);

// Adjoint sensitivities of B returned solutions (Solver::vjp), one launch (mpc_vjp_kernel) in workspace region 0 of ws
// (solve_workspace_doubles(N, B) doubles).  io_aos = 0: state6 [6][B], coeffs [ncoef][B], g_out8 [8][B],
// grad_state6 [6][B], grad_coeffs [ncoef][B], grad_params [8][B]; io_aos = 1: the same per problem ([B][k]).  Always
// field-major: traj, g_traj [8N-2][B], mult [10N-4][B].  g_out8, g_traj, g_obj [B], the gradients and status [B] may be
// null.
struct VjpIO {
  int B = 0, ncoef = 0, io_aos = 0;
  const double *state6 = nullptr, *coeffs = nullptr, *traj = nullptr, *mult = nullptr;
  const double *g_out8 = nullptr, *g_traj = nullptr, *g_obj = nullptr;
  double *grad_state6 = nullptr, *grad_coeffs = nullptr, *grad_params = nullptr;
  int* status = nullptr;
};
// VjpIO plus per-problem cost and model parameters: cost8 [8][B], model4 [4][B] ([B][k] with io_aos), or null for the
// handle's, and grad_model [4][B] (dt, Lf, delta_max, a_max; or null).  A struct of its own so that the kernel instance
// without them keeps VjpIO as its parameter block.
struct VjpCostIO : VjpIO {
  const double* cost8 = nullptr;
  const double* model4 = nullptr;
  double* grad_model = nullptr;
};
cudaError_t launch_vjp(const Params& P, const VjpCostIO& io, double* ws, cudaStream_t stream);

// Forward sensitivities of B returned solutions (Solver::jvp), one launch (mpc_jvp_kernel) in workspace region 0 of ws.
// io_aos = 0: state6 / t_state6 [6][B], coeffs / t_coeffs [ncoef][B], cost8 / t_cost8 [8][B], model4 / t_model4 [4][B],
// t_out8 [8][B]; io_aos = 1: the same per problem ([B][k]).  Always field-major: traj, t_traj [8N-2][B], mult [10N-4][B].
// cost8 / model4 null: the handle's values; a null tangent counts as zero; t_out8, t_traj, t_obj [B] and status [B] may
// be null.
struct JvpIO {
  int B = 0, ncoef = 0, io_aos = 0;
  const double *state6 = nullptr, *coeffs = nullptr, *cost8 = nullptr, *model4 = nullptr, *traj = nullptr, *mult = nullptr;
  const double *t_state6 = nullptr, *t_coeffs = nullptr, *t_cost8 = nullptr, *t_model4 = nullptr;
  double *t_out8 = nullptr, *t_traj = nullptr, *t_obj = nullptr;
  int* status = nullptr;
};
cudaError_t launch_jvp(const Params& P, const JvpIO& io, double* ws, cudaStream_t stream);

// K6 batch I/O: [B][K] <-> [K][B]
cudaError_t launch_aos_to_soa(const double* in, double* out, int B, int K, cudaStream_t stream);
cudaError_t launch_soa_to_aos(const double* in, double* out, int B, int K, cudaStream_t stream);

// K4 polyfit / polyeval, K5 rollout.  aos = 0: field-major arrays ([k][B], what device-resident callers pass);
// aos = 1: the reference's per-problem order ([B][k], what the host entry points receive) -- the kernels index either
// layout themselves, so the host paths need no transpose launches (K6 fused into K4 / K5)
cudaError_t launch_polyfit(const double* xs, const double* ys, int B, int m, int order, double* coeffs,
                           cudaStream_t stream, int aos = 0);
cudaError_t launch_polyeval(const double* coeffs, int ncoef, const double* x, double* y, int B, cudaStream_t stream, int aos = 0);
cudaError_t launch_rollout(const double* state4, const double* act, int B, int H, double dt, double Lf, double* out,
                           cudaStream_t stream, int aos = 0);

// roadmap front-end: pose4 [4][B] (x,y,psi,v global), wp_xy [n_wp][2] -> state6 [6][B], coeffs [4][B] (vehicle frame)
cudaError_t launch_roadmap_reference(const double* pose4, int B, const double* wp_xy, int n_wp, double* state6, double* coeffs,
                                     cudaStream_t stream, int aos = 0);

// DFMA throughput microbenchmark: returns FLOP executed per launch; time it outside.
cudaError_t launch_fp64_peak(double* sink, int blocks, int threads, int iters, cudaStream_t stream, double* flop);
// drcp / ddiv of the sweeps on n operand pairs (device pointers): quot[i] = ddiv(a[i], b[i]), rcp[i] = drcp(b[i])
cudaError_t launch_division_selftest(int n, const double* a, const double* b, double* quot, double* rcp, cudaStream_t stream);

}  // namespace b200mpc
