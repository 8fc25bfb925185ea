// Launchers of the sm_100a kernels behind the C ABI (include/b200mpc.h).  Device pointers only.
#pragma once
#include <cuda_runtime.h>

#include "mpc_core.cuh"

namespace b200mpc {

// doubles of workspace needed to solve B problems at horizon N
size_t solve_workspace_doubles(int N, int B);

// K1+K2+K3 fused: `steps` consecutive interior-point solves per problem (steps > 1 = closed loop, each solve
// starting from the previous solve's predicted state).  All arrays field-major (SoA) over the batch.
//   state6 [6][B], coeffs [ncoef][B], out8 [steps][8][B], traj [8N-2][B] (last step, optional),
//   obj [steps][B] (optional), status [B] (last step, optional), iters [steps][B] (optional)
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
  // batch compaction: after every round from compact_from on, if the unfinished problems fill at most
  // compact_max_live of the occupied workspace slots, they are moved to consecutive slots, so that later rounds run
  // full warps on whole 32-byte sectors (0 = off)
  // adaptive hand-over (automatic rounds only): occupied slots (whole call) at which the cooperative kernel takes over
  int handover_below = 1184;      // one wave of 8 warps on 148 SMs
  int handover_from = 14;         // first round after which it may happen
  int handover_max_rounds = 0;    // 0 = by horizon: 20 up to N = 50, 2 N - 80 above (120 at N = 100); see handover_rounds (solve_kernel.cu)
  double compact_max_live = 0.7;
  int compact_from = 4;
  // pipelined solves (launch_solve_bulk / launch_solve_tail): rounds the tail context runs before its finisher (0 = by
  // horizon: 10 up to N = 50, 2 N - 80 above)
  int tail_rounds = 0;
  int tail_take_below = 0;   // long horizons: occupied slots at which the cooperative kernel takes a tail over (0 = 32)
  bool coop = true;       // latency path = cooperative warp-per-problem kernel (false: thread-per-problem fused kernel)
};
struct SplitStreams {   // auxiliary streams / events owned by the handle (n_aux <= 3)
  int n_aux = 0;
  cudaStream_t aux[3] = {nullptr, nullptr, nullptr};
  cudaEvent_t fork = nullptr, join[3] = {nullptr, nullptr, nullptr};
};
cudaError_t launch_solve(const Params& P, int B, int steps, const double* state6, const double* coeffs, int ncoef,
                         double* ws, double* out8, double* traj, double* obj, int* status, int* iters,
                         const SolveConfig& cfg, cudaStream_t stream, const SplitStreams* ss, long long* n_launches,
                         int io_aos = 0);   // io_aos = 1: state6 [B][6], coeffs [B][ncoef], out8 [steps][B][8] (reference order)

// Pipelined solves: one solve as two launch sequences (see solve_kernel.cu).  A tail context is a workspace of
// solve_workspace_doubles(N, slots) doubles.
struct TailCtx {
  double* ws = nullptr;
  int slots = 0;
};
cudaError_t launch_solve_bulk(const Params& P, int B, const double* state6, const double* coeffs, int ncoef, double* ws, double* out8,
                              double* traj, double* obj, int* status, int* iters, const SolveConfig& cfg, cudaStream_t stream,
                              long long* n_launches, int io_aos, const TailCtx& tail);
cudaError_t launch_solve_tail(const Params& P, int B, const double* state6, const double* coeffs, int ncoef, double* out8, double* traj,
                              double* obj, int* status, int* iters, const SolveConfig& cfg, cudaStream_t stream, long long* n_launches,
                              int io_aos, const TailCtx& tail);

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
