// Interior-point solve kernels for sm_100a (K1 derivative evaluation, K2 Riccati KKT solve, K3 barrier / line
// search / filter / convergence logic).  Replaces CppAD::ipopt::solve at
// /root/reference/mpc_to_line/solution/MPC.cpp:241-243.
//
// Throughput path (mpc_core.cuh): one problem per thread; every per-problem vector lives in a warp-interleaved HBM
// workspace (each workspace access of a warp is one coalesced 256-byte row) and the 7x7 Riccati blocks live in
// registers.  One interior-point iteration = three sweeps over the horizon, each its own kernel
//   init | factor | forward | step        launched round after round on one stream (replayed as one CUDA graph),
// with its own register budget (the Riccati factorisation needs ~250 registers, the step sweep ~240 with its
// stage-to-stage values in registers, the forward sweep 168) and a small instruction footprint.
// Between rounds mpc_repack_kernel compacts the problems that are still iterating into consecutive workspace slots
// (second workspace region, slot -> problem map, level state in device memory), so late rounds run full warps.
// Latency path (mpc_coop.cuh): one problem per warp, lane <-> stage.  mpc_coop_kernel finishes whatever is still
// iterating once the compacted batch fits one of its waves (or after the last round) and solves small batches on its own.
// mpc_fused_kernel loops the three thread-per-problem sweeps in one launch (comparison / fallback for horizons whose
// per-stage scratch does not fit the cooperative kernel's shared memory).
#include <type_traits>

#include "kernels.h"
#include "mpc_coop.cuh"

namespace b200mpc {

constexpr int kBlock = 64;
// resident blocks per SM the light sweeps are compiled for (register cap = 65536 / (64 * blocks)).
// The step sweep runs at 4 blocks per SM: 228 registers, nothing spilled.  At 6 blocks (168 registers, 240 B of spill
// stores and 352 B of spill loads per thread and stage) it is 3 % slower with one caller and with overlapped callers
// (profiles/r2_sweep_tuning_ab.json, r2_sb*: 13.59 -> 14.05 M solves/s; 5 blocks: 13.57 M) -- the sweep is bound by
// its dependent instruction chains, not by the number of resident warps.
constexpr int kFwdBlocks = 6, kStepBlocks = 4, kFactorBlocks = 4;

// One workspace region holds every problem of a batch; the buffer the handle allocates has two of them (the batch
// compaction moves the unfinished problems back and forth), two slot -> problem maps and the counters.
constexpr int kMaxParts = 4;
// per-part compaction state in device memory (ints)
enum Desc { kLevel = 0, kCount, kLive, kAlloc, kTicket, kHanded, kDescInts = 8 };
static size_t region_doubles(int N, int B) {
  size_t groups = ((size_t)B + 31) / 32;
  return groups * (size_t)workspace_doubles_per_problem(N) * 32;
}
static size_t aux_doubles(int B) { return ((size_t)B + 1) / 2 * 2 + kMaxParts * kDescInts; }   // 2 int maps + state
size_t solve_workspace_doubles(int N, int B) { return 2 * region_doubles(N, B) + aux_doubles(B); }
// the parts of a buffer of solve_workspace_doubles(N, B) doubles: region 0 | region 1 | map 0 | map 1 | compaction state
struct WsLayout {
  double* ws0;
  double* ws1;
  int* map0;
  int* map1;
  int* desc;
};
static WsLayout ws_layout(double* ws, int N, int B) {
  const size_t reg = region_doubles(N, B);
  int* ints = reinterpret_cast<int*>(ws + 2 * reg);
  const size_t map_ints = ((size_t)B + 1) / 2 * 2;
  return WsLayout{ws, ws + reg, ints, ints + map_ints, ints + 2 * map_ints};
}

struct SolveArgs {
  int B, steps, step, ncoef;
  int io_aos;             // layout of state6 / coeffs / out8: 0 = field-major [k][B] (device callers), 1 = the reference's
                          // per-problem order [B][k] (host entry points: no separate transpose kernels, K6 is fused here)
  int b0, b1;             // this launch covers problems [b0, b1) of the B-problem batch (B stays the array stride)
  int warm;               // closed loop: steps > 0 start from the shifted previous solution
  double mu_warm;
  const double* state6;   // [6][B]
  const double* coeffs;   // [ncoef][B]
  double* ws;             // workspace region 0: slot == problem (level 0)
  // batch compaction (desc == null: off).  Level k >= 1 lives in region k & 1 with the slot -> problem map (k - 1) & 1;
  // desc = {level, occupied slots, live problems counted by the step kernel, slot allocator, block ticket}
  double* ws1;
  int* map0;
  int* map1;
  int* desc;
  int count_live;         // step kernel: count the problems that are not finished (a compaction attempt follows)
  double* out8;           // [steps][8][B]
  double* traj;           // [8N-2][B] or null (last step)
  double* obj;            // [steps][B] or null
  int* status;            // [B] or null (last step)
  int* iters;             // [steps][B] or null
  const double* x_init;   // [8N-2][B] or null: fresh solves start from this point (Solver::init_guess)
  const double* mult_init;   // [10N-4][B] or null (with x_init)
  double mu_init;
  double* mult;           // [10N-4][B] or null (last step)
};

// Per-problem rows (b200mpc_solve_batch_cost*, b200mpc_solve_batch_model*): the kernel instances with ROWS != kNoRows
// take this parameter block, every other instance SolveArgs, whose layout (and so the machine code of those instances)
// does not change.  kCostRows instances read cost8 only; kModelRows instances read model4 and, if given, cost8.  They are
// kept apart because per-problem dt, Lf and bounds (registers instead of the handle's constants) change the code of the
// sweeps, and the cost rows alone must not pay for that.
enum Rows { kNoRows = 0, kCostRows = 1, kModelRows = 2 };
struct CostArgs : SolveArgs {
  const double* cost8;    // [8][B] ([B][8] with io_aos) or null: ref_v, w_cte, w_epsi, w_v, w_delta, w_a, w_ddelta, w_da
  const double* model4;   // [4][B] ([B][4] with io_aos) or null: dt, Lf, delta_max, a_max
};
template <int ROWS>
using ArgsT = typename std::conditional<ROWS != kNoRows, CostArgs, SolveArgs>::type;

__device__ __forceinline__ double* slot_base(const Params& P, double* ws, int slot) {
  return ws + (size_t)(slot >> 5) * (size_t)workspace_doubles_per_problem(P.N) * 32 + (slot & 31);
}
// thread (or warp) i of a launch -> workspace slot (+ its region) and problem index; false: nothing to do
__device__ __forceinline__ bool locate(const SolveArgs& A, int i, int& slot, int& b, double*& ws, bool sweeps = true) {
  slot = A.b0 + i;
  const int level = A.desc ? A.desc[kLevel] : 0;
  if (sweeps && level > 0 && A.desc[kHanded]) return false;   // the cooperative kernel has taken the rest over
  if (level == 0) {
    if (slot >= A.b1) return false;
    b = slot; ws = A.ws;
  } else {
    if (i >= A.desc[kCount]) return false;
    b = ((level & 1) ? A.map0 : A.map1)[slot];
    ws = (level & 1) ? A.ws1 : A.ws;
  }
  return true;
}
__device__ __forceinline__ void load_coeffs(const SolveArgs& A, int b, double* cf) {
  const size_t sb = A.io_aos ? (size_t)A.ncoef : 1, sk = A.io_aos ? 1 : (size_t)A.B;
#pragma unroll
  for (int i = 0; i < kMaxCoef; ++i) cf[i] = i < A.ncoef ? A.coeffs[(size_t)b * sb + (size_t)i * sk] : 0.0;
}
// element k of the returned 8-vector of problem b at closed-loop step `step`
__device__ __forceinline__ size_t out8_index(const SolveArgs& A, int step, int k, int b) {
  return (size_t)step * 8 * A.B + (A.io_aos ? (size_t)b * 8 + k : (size_t)k * A.B + b);
}
// initial state of closed-loop step `step`: the caller's state for step 0, else the previous step's out8[0..5]
// (solution/main.cpp:66)
__device__ __forceinline__ void load_state6(const SolveArgs& A, int b, double* s0) {
#pragma unroll
  for (int k = 0; k < 6; ++k)
    s0[k] = A.step == 0 ? A.state6[A.io_aos ? (size_t)b * 6 + k : (size_t)k * A.B + b] : A.out8[out8_index(A, A.step - 1, k, b)];
}
// Problem b's row of cost8 (layout io_aos) over the eight cost fields of Q, which is a copy of the handle's Params.  The
// row is indexed by problem, not by workspace slot, like the coefficients, so compaction and hand-offs need nothing.
// False: a non-finite entry (Q is left unchanged then).
__device__ __forceinline__ bool cost_row(const double* cost8, int io_aos, int B, int b, Params& Q) {
  double c[8];
  bool ok = true;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    c[k] = cost8[io_aos ? (size_t)b * 8 + k : (size_t)k * B + b];
    ok &= fabs(c[k]) <= DBL_MAX;
  }
  if (ok) {
    Q.ref_v = c[0]; Q.w_cte = c[1]; Q.w_epsi = c[2]; Q.w_v = c[3];
    Q.w_delta = c[4]; Q.w_a = c[5]; Q.w_ddelta = c[6]; Q.w_da = c[7];
  }
  return ok;
}
// Problem b's row of model4 over dt, Lf, delta_max, a_max of Q, and Q's derived constants recomputed.  False: an entry
// that is not finite and positive, what b200mpc_create rejects for a handle (Q is left unchanged then).
__device__ __forceinline__ bool model_row(const double* model4, int io_aos, int B, int b, Params& Q) {
  double c[4];
  bool ok = true;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    c[k] = model4[io_aos ? (size_t)b * 4 + k : (size_t)k * B + b];
    ok &= c[k] > 0.0 && c[k] <= DBL_MAX;
  }
  if (ok) {
    Q.dt = c[0]; Q.Lf = c[1]; Q.delta_max = c[2]; Q.a_max = c[3];
    Q.finalize();
  }
  return ok;
}
// Per-problem instances: the solver of problem b runs on Q with b's rows (kModelRows: model4 and cost8 if given).  An
// invalid row makes ref_v NaN, so the objective at the start point is NaN and the start-point check stops the problem
// with status -13 and 0 iterations (Solver::init_finish / guess_check), as for a non-finite x_init; the later sweeps
// never see it.
template <int ROWS>
__device__ __forceinline__ void load_cost(const ArgsT<ROWS>& A, int b, Params& Q) {
  if constexpr (ROWS == kCostRows) {
    if (!cost_row(A.cost8, A.io_aos, A.B, b, Q)) Q.ref_v = NAN;
  } else if constexpr (ROWS == kModelRows) {
    bool ok = !A.cost8 || cost_row(A.cost8, A.io_aos, A.B, b, Q);
    ok &= model_row(A.model4, A.io_aos, A.B, b, Q);
    if (!ok) Q.ref_v = NAN;
  }
}

// Warm-start I/O (SolveArgs::x_init / mult_init / mult) is compiled only into the WIO = true instance of each kernel that
// starts or finishes problems, and that instance is launched only when a call uses it: a call without it runs kernels
// that do not carry its code (the factor and step sweeps: the same machine code as without the feature).
template <bool WIO>
__device__ __forceinline__ void write_result(const Params& P, const SolveArgs& A, int b, Solver<32>& S) {
  Result R;
  S.finish(R, (A.traj && A.step == A.steps - 1) ? A.traj + b : nullptr, (size_t)A.B);
#pragma unroll
  for (int k = 0; k < 8; ++k) A.out8[out8_index(A, A.step, k, b)] = R.out8[k];
  if (A.obj) A.obj[(size_t)A.step * A.B + b] = R.obj;
  if (A.iters) A.iters[(size_t)A.step * A.B + b] = R.iters;
  if (A.status && A.step == A.steps - 1) A.status[b] = R.status;
  if (WIO && A.mult && A.step == A.steps - 1) S.write_mult(A.mult + b, (size_t)A.B);
}
// the caller's multipliers of problem b for a fresh solve from its point (slot == problem), or null
__device__ __forceinline__ const double* guess_mult(const SolveArgs& A, int b) { return A.mult_init ? A.mult_init + b : nullptr; }

// one atomic per group of converged lanes
__device__ __forceinline__ void count_live(int* counter) {
  const unsigned m = __activemask();
  if ((int)(threadIdx.x & 31) == __ffs(m) - 1) atomicAdd(counter, __popc(m));
}

// ---- per-pass kernels ---------------------------------------------------------------------------------------
template <bool WIO, int ROWS>
__global__ void __launch_bounds__(kBlock) mpc_init_kernel(const __grid_constant__ Params P, const __grid_constant__ ArgsT<ROWS> A) {
  const int b = A.b0 + blockIdx.x * blockDim.x + threadIdx.x;   // always launched on the uncompacted batch
  if (b >= A.b1) return;
  if (b == A.b0 && A.desc)
    for (int k = 0; k < kDescInts; ++k) A.desc[k] = 0;
  Params Q = P;
  load_cost<ROWS>(A, b, Q);
  Solver<32> S(ROWS ? Q : P, slot_base(P, A.ws, b), b & 31);
  double s0[6], cf[kMaxCoef];
  load_state6(A, b, s0);
  load_coeffs(A, b, cf);
  const bool cold = !(A.warm && A.step > 0) && !(WIO && A.x_init);
  if (A.warm && A.step > 0) { S.set_coeffs(cf, A.ncoef); S.init_warm(s0, A.mu_warm); }
  else if (WIO && A.x_init) { S.set_coeffs(cf, A.ncoef); S.init_guess(s0, A.x_init + b, (size_t)A.B, guess_mult(A, b), (size_t)A.B, A.mu_init); }
  else S.init(s0, cf, A.ncoef);
  S.store_state();
  if (cold && S.phase == PH_FACTOR) S.kernel_ls_round(s0);   // the sweeps start at the first Newton round
  if (S.phase == PH_DONE) write_result<WIO>(P, A, b, S);   // invalid number at the starting point, or converged there
}

template <bool WIO, int ROWS>
__global__ void __launch_bounds__(kBlock, kFactorBlocks) mpc_factor_kernel(const __grid_constant__ Params P, const __grid_constant__ ArgsT<ROWS> A) {
  int slot, b;
  double* ws;
  if (!locate(A, blockIdx.x * blockDim.x + threadIdx.x, slot, b, ws)) return;
  Params Q = P;
  Solver<32> S(ROWS ? Q : P, slot_base(P, ws, slot), slot & 31);
  if (S.load_phase() != PH_FACTOR) return;
  load_cost<ROWS>(A, b, Q);
  __shared__ double stage[2 * kStageVals * kBlock];   // [buffer][value][thread]
  S.sb = stage + threadIdx.x; S.sbs = kBlock;
  load_coeffs(A, b, S.cf);
  S.kernel_factor();
  if (S.phase == PH_DONE) {   // inertia correction exhausted (IpPDPerturbationHandler.cpp:380-388)
    S.load_state();
    write_result<WIO>(P, A, b, S);
  }
}

template <int ROWS>
__global__ void __launch_bounds__(kBlock, kFwdBlocks) mpc_forward_kernel(const __grid_constant__ Params P, const __grid_constant__ ArgsT<ROWS> A) {
  int slot, b;
  double* ws;
  if (!locate(A, blockIdx.x * blockDim.x + threadIdx.x, slot, b, ws)) return;
  Params Q = P;
  Solver<32> S(ROWS ? Q : P, slot_base(P, ws, slot), slot & 31);
  if (S.load_phase() != PH_FORWARD) return;
  load_cost<ROWS>(A, b, Q);
  load_coeffs(A, b, S.cf);
  S.kernel_forward();
}

template <bool WIO, int ROWS>
__global__ void __launch_bounds__(kBlock, kStepBlocks) mpc_step_kernel(const __grid_constant__ Params P, const __grid_constant__ ArgsT<ROWS> A) {
  int slot, b;
  double* ws;
  if (!locate(A, blockIdx.x * blockDim.x + threadIdx.x, slot, b, ws)) return;
  Params Q = P;
  Solver<32> S(ROWS ? Q : P, slot_base(P, ws, slot), slot & 31);
  const int ph = S.load_phase();
  if (ph != PH_STEP) {
    if (A.count_live && ph != PH_DONE) count_live(A.desc + kLive);
    return;
  }
  load_cost<ROWS>(A, b, Q);
  double carry[kCarry];
  S.cr = carry; S.cs = 1;
  __shared__ double stage[2 * kStepStageVals * kBlock];   // [buffer][value][thread]
  S.sb = stage + threadIdx.x; S.sbs = kBlock;
  load_coeffs(A, b, S.cf);
  S.kernel_step();
  if (S.phase == PH_DONE) write_result<WIO>(P, A, b, S);
  else if (A.count_live) count_live(A.desc + kLive);
}

// ---- batch compaction ------------------------------------------------------------------------------------------
// Runs after a step kernel that counted the live (unfinished) problems.  If they fill at most `max_live` of the
// occupied slots they move to consecutive slots of the other region (level + 1); the following launches find the new
// level in desc.  The running lanes of a warp take consecutive destination slots, so the rows they write are
// contiguous; the slot order among warps is first come, first served (results do not depend on the slot a problem
// sits in).  The last block to finish commits the new level and clears the counters.
// Tail hand-off (pipelined solves, launch_solve_bulk / launch_solve_tail): with export_below > 0 the kernel moves the live
// problems OUT of this workspace as soon as at most export_below are left -- into region 1 of a small tail context
// (T.ws1, slot -> problem map T.map0, level 1 in T.desc) -- and leaves this workspace empty (level >= 1, no occupied
// slots: every later launch on it finds nothing to do).  The tail context is finished by its own launches while the
// next batch already runs in this workspace.
__global__ void __launch_bounds__(256) mpc_repack_kernel(const __grid_constant__ Params P, const __grid_constant__ SolveArgs A,
                                                         double max_live, int export_below, double* t_ws1, int* t_map0, int* t_desc) {
  int* desc = A.desc;
  const int level = desc[kLevel], live_n = desc[kLive];
  const int occupied = level == 0 ? A.b1 - A.b0 : desc[kCount];
  const bool exp = export_below > 0 && live_n > 0 && live_n <= export_below;
  const bool go = exp || (live_n > 0 && (double)live_n <= max_live * (double)occupied);
  if (go) {
    int slot = 0, b = 0;
    double* ws = A.ws;
    const bool in = locate(A, blockIdx.x * blockDim.x + threadIdx.x, slot, b, ws);
    const Ws<32> src{slot_base(P, ws, slot), slot & 31};
    const bool live = in && (int)src(iPHASE) != PH_DONE;
    const unsigned m = __ballot_sync(0xffffffffu, live);
    const int lane = threadIdx.x & 31;
    int base = 0;
    if (m != 0 && lane == 0) base = atomicAdd(desc + kAlloc, __popc(m));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (live) {
      const int rank = base + __popc(m & ((1u << lane) - 1u));
      if (exp) {
        t_map0[rank] = b;
        repack_problem(P, src, Ws<32>{slot_base(P, t_ws1, rank), rank & 31});
      } else {
        const int ds = A.b0 + rank;
        (((level + 1) & 1) ? A.map0 : A.map1)[ds] = b;
        repack_problem(P, src, Ws<32>{slot_base(P, ((level + 1) & 1) ? A.ws1 : A.ws, ds), ds & 31});
      }
    }
  }
  __syncthreads();   // every thread of the block has read desc
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(desc + kTicket, 1) == (int)gridDim.x - 1) {
      if (exp) {
        t_desc[kLevel] = 1; t_desc[kCount] = desc[kAlloc];
        desc[kCount] = 0; desc[kLevel] = level > 0 ? level : 1;
      } else if (go) { desc[kCount] = desc[kAlloc]; desc[kLevel] = level + 1; }
      desc[kLive] = 0; desc[kAlloc] = 0; desc[kTicket] = 0;
    }
  }
}
// an empty tail context: level 1 with no occupied slots (level 0 would mean "slot == problem" for every slot)
__global__ void mpc_tail_reset_kernel(int* t_desc) {
  if (threadIdx.x < kDescInts) t_desc[threadIdx.x] = threadIdx.x == kLevel ? 1 : 0;
}

// ---- fused kernel: finishes whatever is still active (fresh == 1: starts from the inputs) ---------------------
template <bool WIO, int ROWS>
__global__ void __launch_bounds__(kBlock) mpc_fused_kernel(const __grid_constant__ Params P, const __grid_constant__ ArgsT<ROWS> A, int fresh) {
  int slot, b;
  double* ws;
  if (!locate(A, blockIdx.x * blockDim.x + threadIdx.x, slot, b, ws, false)) return;
  Params Q = P;
  load_cost<ROWS>(A, b, Q);
  Solver<32> S(ROWS ? Q : P, slot_base(P, ws, slot), slot & 31);
  double carry[kCarry];
  S.cr = carry; S.cs = 1;
  load_coeffs(A, b, S.cf);
  if (fresh) {
    double s0[6];
    load_state6(A, b, s0);
    if (A.warm && A.step > 0) S.init_warm(s0, A.mu_warm);
    else if (WIO && A.x_init) S.init_guess(s0, A.x_init + b, (size_t)A.B, guess_mult(A, b), (size_t)A.B, A.mu_init);
    else S.init(s0, S.cf, kMaxCoef);
  } else {
    if (S.load_phase() == PH_DONE) return;
    S.load_state();
  }
  while (S.phase != PH_DONE) S.trip();
  S.store_state();
  write_result<WIO>(P, A, b, S);
}

// ---- cooperative kernel: one problem per warp (latency path: small batches, the tail of a batch, stragglers) -----
struct DevExec {
  int lane;
  __device__ __forceinline__ bool lane0() const { return lane == 0; }
  __device__ __forceinline__ void sync() const { __syncwarp(); }
  template <class F>
  __device__ __forceinline__ void for_stages(int n, F f) const {
    for (int t = lane; t < n; t += 32) f(t);
  }
};

// take_below > 0: conditional hand-over after a round -- the kernel acts only once the batch has been compacted to at
// most take_below occupied slots (two waves of the cooperative kernel); from then on the sweeps of later rounds find
// nothing to do
template <bool WIO, int ROWS>
__global__ void __launch_bounds__(128) mpc_coop_kernel(const __grid_constant__ Params P, const __grid_constant__ ArgsT<ROWS> A, int fresh,
                                                       int warps_per_block, int doubles_per_warp, int take_below) {
  extern __shared__ double coop_smem[];
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (take_below > 0) {
    if (!A.desc || A.desc[kLevel] == 0 || A.desc[kCount] > take_below) return;
    if (threadIdx.x == 0) A.desc[kHanded] = 1;   // only the sweeps read it
  }
  if (wib >= warps_per_block) return;
  double* mine = coop_smem + (size_t)wib * doubles_per_warp;
  CoopStage* st = reinterpret_cast<CoopStage*>(mine);
  CoopPub* pub = reinterpret_cast<CoopPub*>(mine + (size_t)P.N * kCoopStageDoubles);
  // one problem per warp at a time; the grid is capped at a few waves and every warp walks on through the slots (a
  // launch that finds little or nothing to do must not cost thousands of 100 KB-shared-memory blocks)
  for (int idx = blockIdx.x * warps_per_block + wib;; idx += gridDim.x * warps_per_block) {
    int slot, b;
    double* ws;
    if (!locate(A, idx, slot, b, ws, false)) return;
    Params Q = P;
    load_cost<ROWS>(A, b, Q);
    Solver<32> S(ROWS ? Q : P, slot_base(P, ws, slot), slot & 31);
    load_coeffs(A, b, S.cf);
    CoopSolver<32, DevExec> C(S, st, pub, DevExec{lane});
    if (fresh) {
      double s0[6];
      load_state6(A, b, s0);
      if (A.warm && A.step > 0) C.init_warm(s0, A.mu_warm);
      else if (WIO && A.x_init) C.init_guess(s0, A.x_init + b, (size_t)A.B, guess_mult(A, b), (size_t)A.B, A.mu_init);
      else C.init(s0);
    } else {
      if (S.load_phase() == PH_DONE) continue;   // whole warp
      if (lane == 0) S.load_state();
      __syncwarp();
    }
    C.run();
    if (lane == 0) {
      S.store_state();
      write_result<WIO>(P, A, b, S);
    }
    __syncwarp();
  }
}

constexpr size_t kCoopSmemMax = 200 * 1024;   // dynamic shared memory of one cooperative block, at most
// per-device, once (b200mpc_create)
cudaError_t solver_prepare_device() {
  cudaError_t e = cudaFuncSetAttribute(mpc_coop_kernel<false, kNoRows>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kCoopSmemMax);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(mpc_coop_kernel<true, kNoRows>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kCoopSmemMax);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(mpc_coop_kernel<true, kCostRows>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kCoopSmemMax);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(mpc_coop_kernel<true, kModelRows>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kCoopSmemMax);
  return e;
}

static size_t coop_doubles_per_warp(int N) { return (size_t)N * kCoopStageDoubles + (sizeof(CoopPub) + 7) / 8; }
// block of the cooperative kernel at horizon N: up to 4 problems (warps), per-problem scratch in shared memory;
// warps = 0: the horizon does not fit
struct CoopShape {
  int warps;
  size_t smem;
};
static CoopShape coop_shape(int N) {
  const size_t per_warp = coop_doubles_per_warp(N) * sizeof(double);
  if (per_warp > kCoopSmemMax) return CoopShape{0, 0};
  int wpb = (int)(kCoopSmemMax / per_warp);
  if (wpb > 4) wpb = 4;
  return CoopShape{wpb, per_warp * wpb};
}
// warps of the cooperative kernel that are resident on the device at once (0: the horizon does not fit), 2 blocks per SM
// by registers
static int coop_resident_warps(int N) {
  const CoopShape c = coop_shape(N);
  if (c.warps == 0) return 0;
  const int wpb = c.warps;
  int blocks = (int)((size_t)227 * 1024 / c.smem);
  if (blocks > 2) blocks = 2;
  int sms = 148;
  int dev = 0;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  return sms * blocks * wpb;
}

// the kernels' parameter block for problems [b0, b1) of the B-problem batch in workspace L (desc: the compaction state
// of these problems, or null: no compaction); warm_mu > 0: closed-loop steps after the first start from the shifted
// previous solution with this barrier parameter
static CostArgs solve_args(int B, int steps, const SolveIO& io, const WsLayout& L, int* desc, int b0, int b1, double warm_mu) {
  CostArgs A{};
  A.B = B; A.steps = steps; A.ncoef = io.ncoef; A.io_aos = io.io_aos ? 1 : 0; A.b0 = b0; A.b1 = b1;
  A.warm = warm_mu > 0.0 ? 1 : 0; A.mu_warm = warm_mu;
  A.state6 = io.state6; A.coeffs = io.coeffs;
  A.ws = L.ws0; A.ws1 = L.ws1; A.map0 = L.map0; A.map1 = L.map1; A.desc = desc;
  A.out8 = io.out8; A.traj = io.traj; A.obj = io.obj; A.status = io.status; A.iters = io.iters;
  A.x_init = io.x_init; A.mult_init = io.mult_init; A.mu_init = io.mu_init; A.mult = io.mult;
  A.cost8 = io.cost8; A.model4 = io.model4;
  return A;
}

static int sweep_grid(const SolveArgs& A) { return (A.b1 - A.b0 + kBlock - 1) / kBlock; }
// the call reads a start point or writes multipliers: the WIO = true kernel instances.  A call with per-problem cost or
// model rows runs the <true, kCostRows> or <true, kModelRows> instances (null x_init / mult do nothing there); the others
// get the SolveArgs part of A.
static bool warm_io(const SolveArgs& A) { return A.x_init != nullptr || A.mult != nullptr; }
static int rows_of(const CostArgs& A) { return A.model4 ? kModelRows : (A.cost8 ? kCostRows : kNoRows); }
static void launch_init(const Params& P, const CostArgs& A, cudaStream_t stream, long long* n) {
  if (rows_of(A) == kModelRows) mpc_init_kernel<true, kModelRows><<<sweep_grid(A), kBlock, 0, stream>>>(P, A);
  else if (rows_of(A) == kCostRows) mpc_init_kernel<true, kCostRows><<<sweep_grid(A), kBlock, 0, stream>>>(P, A);
  else if (warm_io(A)) mpc_init_kernel<true, kNoRows><<<sweep_grid(A), kBlock, 0, stream>>>(P, A);
  else mpc_init_kernel<false, kNoRows><<<sweep_grid(A), kBlock, 0, stream>>>(P, A);
  *n += 1;
}

template <int R>
static void launch_round_rows(const Params& P, const CostArgs& A, const CostArgs& As, cudaStream_t stream) {
  mpc_factor_kernel<true, R><<<sweep_grid(A), kBlock, 0, stream>>>(P, A);
  mpc_forward_kernel<R><<<sweep_grid(A), kBlock, 0, stream>>>(P, A);
  mpc_step_kernel<true, R><<<sweep_grid(A), kBlock, 0, stream>>>(P, As);
}

// The launch helpers add one to *n per kernel they launch.  launch_round: one round of the thread-per-problem sweeps;
// count_live: the step kernel counts the unfinished problems for the compaction attempt that follows
static void launch_round(const Params& P, const CostArgs& A, bool count_live, cudaStream_t stream, long long* n) {
  CostArgs As = A;
  As.count_live = count_live ? 1 : 0;
  if (rows_of(A) == kModelRows) {
    launch_round_rows<kModelRows>(P, A, As, stream);
  } else if (rows_of(A) == kCostRows) {
    launch_round_rows<kCostRows>(P, A, As, stream);
  } else {
    if (warm_io(A)) mpc_factor_kernel<true, kNoRows><<<sweep_grid(A), kBlock, 0, stream>>>(P, A);
    else mpc_factor_kernel<false, kNoRows><<<sweep_grid(A), kBlock, 0, stream>>>(P, A);
    mpc_forward_kernel<kNoRows><<<sweep_grid(A), kBlock, 0, stream>>>(P, A);
    if (warm_io(A)) mpc_step_kernel<true, kNoRows><<<sweep_grid(A), kBlock, 0, stream>>>(P, As);
    else mpc_step_kernel<false, kNoRows><<<sweep_grid(A), kBlock, 0, stream>>>(P, As);
  }
  *n += 3;
}

// a compaction attempt after a counting round; export_below > 0: a hand-off to the tail context T (mpc_repack_kernel)
static void launch_repack(const Params& P, const SolveArgs& A, double max_live, cudaStream_t stream, long long* n,
                          int export_below = 0, const WsLayout& T = WsLayout{}) {
  mpc_repack_kernel<<<(A.b1 - A.b0 + 255) / 256, 256, 0, stream>>>(P, A, max_live, export_below, T.ws1, T.map0, T.desc);
  *n += 1;
}

static void launch_fused(const Params& P, const CostArgs& A, int fresh, cudaStream_t stream, long long* n) {
  if (rows_of(A) == kModelRows) mpc_fused_kernel<true, kModelRows><<<sweep_grid(A), kBlock, 0, stream>>>(P, A, fresh);
  else if (rows_of(A) == kCostRows) mpc_fused_kernel<true, kCostRows><<<sweep_grid(A), kBlock, 0, stream>>>(P, A, fresh);
  else if (warm_io(A)) mpc_fused_kernel<true, kNoRows><<<sweep_grid(A), kBlock, 0, stream>>>(P, A, fresh);
  else mpc_fused_kernel<false, kNoRows><<<sweep_grid(A), kBlock, 0, stream>>>(P, A, fresh);
  *n += 1;
}

// launches the cooperative kernel if the horizon fits in shared memory (*err: the launch's error); returns false otherwise
static bool launch_coop(const Params& P, const CostArgs& A, int fresh, int take_below, cudaStream_t stream, cudaError_t* err,
                        long long* n) {
  const CoopShape c = coop_shape(P.N);
  if (c.warps == 0) return false;
  const int wpb = c.warps;
  const int nb = take_below > 0 && take_below < A.b1 - A.b0 ? take_below : A.b1 - A.b0;
  int grid = (nb + wpb - 1) / wpb;
  const int cap = 4 * coop_resident_warps(P.N) / wpb;   // four waves; the warps stride over the rest
  if (cap > 0 && grid > cap) grid = cap;
  // no idle warps: their registers would stay allocated
  const int dpw = (int)coop_doubles_per_warp(P.N);
  if (rows_of(A) == kModelRows) mpc_coop_kernel<true, kModelRows><<<grid, 32 * wpb, c.smem, stream>>>(P, A, fresh, wpb, dpw, take_below);
  else if (rows_of(A) == kCostRows) mpc_coop_kernel<true, kCostRows><<<grid, 32 * wpb, c.smem, stream>>>(P, A, fresh, wpb, dpw, take_below);
  else if (warm_io(A)) mpc_coop_kernel<true, kNoRows><<<grid, 32 * wpb, c.smem, stream>>>(P, A, fresh, wpb, dpw, take_below);
  else mpc_coop_kernel<false, kNoRows><<<grid, 32 * wpb, c.smem, stream>>>(P, A, fresh, wpb, dpw, take_below);
  *n += 1;
  *err = cudaGetLastError();
  return true;
}

// rounds of the thread-per-problem sweeps after which the cooperative kernel takes every remaining problem over.
// Longer horizons have a longer tail of iteration counts (N = 100: 3.6 % of the problems need more than 20, 1.8 % more
// than 100) and a slower cooperative kernel (0.34 ms per problem and iteration at N = 100, 2 warps per SM), so the sweeps
// keep the tail longer there: measured with 4 overlapped batches of 65 536 problems at N = 100, 20 rounds 267 ms per
// batch, 120 rounds 225 ms; N <= 50 does not gain (profiles/r1_handover_sweep_long_horizons.log).
static int handover_rounds(const Params& P) { return P.N <= 50 ? 20 : 2 * P.N - 80; }

// launches every kernel of the solve of problems [b0, b1) on one stream
static cudaError_t launch_part(const Params& P, CostArgs A, const SolveConfig& cfg, int rounds, int take_below, cudaStream_t stream, long long* n) {
  for (int step = 0; step < A.steps; ++step) {
    A.step = step;
    cudaError_t ce = cudaSuccess;
    if (cfg.mode == kModeFused || A.B < cfg.fused_below) {
      A.desc = nullptr;
      if (!(cfg.coop && cfg.mode != kModeFused && launch_coop(P, A, 1, 0, stream, &ce, n))) launch_fused(P, A, 1, stream, n);
    } else {
      launch_init(P, A, stream, n);
      for (int r = 0; r < rounds; ++r) {
        // a compaction attempt follows every round from compact_from on (not the last: only the finisher is left)
        const bool attempt = A.desc && r + 1 >= cfg.compact_from && r + 1 < rounds;
        launch_round(P, A, attempt, stream, n);
        if (!attempt) continue;
        launch_repack(P, A, cfg.compact_max_live, stream, n);
        if (take_below > 0 && r + 1 >= cfg.handover_from && cfg.coop) launch_coop(P, A, 0, take_below, stream, &ce, n);
        if (ce != cudaSuccess) return ce;
      }
      if (!(cfg.coop && launch_coop(P, A, 0, 0, stream, &ce, n))) launch_fused(P, A, 0, stream, n);
    }
    if (ce == cudaSuccess) ce = cudaGetLastError();
    if (ce != cudaSuccess) return ce;
  }
  return cudaSuccess;
}

// A large batch is cut into `split` contiguous parts that run concurrently on the caller's stream and on auxiliary
// streams (fork / join with events; capturable into a CUDA graph): the kernels of different parts are in different
// sweeps at any moment, which fills the partial waves of the 252-register factor kernel and hides the thin tail of
// one part behind the bulk of another even when the caller uses a single stream.
cudaError_t launch_solve(const Params& P, int B, int steps, const SolveIO& io, double* ws, const SolveConfig& cfg,
                         cudaStream_t stream, const SplitStreams* ss, long long* n) {
  if (B <= 0) return cudaSuccess;
  const WsLayout L = ws_layout(ws, P.N, B);   // the compaction state holds one record per part
  // a warm-started step reads the previous solution at the problem's own slot: no compaction then
  int* desc = (!(cfg.compact_max_live > 0.0) || cfg.warm_start) ? nullptr : L.desc;
  int parts = 1;
  if (ss && cfg.mode == kModePerPass && cfg.split > 1 && B >= cfg.split * cfg.fused_below) parts = cfg.split < ss->n_aux + 1 ? cfg.split : ss->n_aux + 1;
  // automatic setting: up to handover_rounds() rounds, and after every late round the cooperative kernel takes the
  // rest over as soon as the compacted batch fits its two waves (the launches after that find nothing to do); a fixed
  // number of rounds (b200mpc_set_solver_mode) hands over exactly there
  const bool adaptive = cfg.rounds <= 0 && desc != nullptr && cfg.coop && cfg.handover_below > 0;
  const int rounds = cfg.rounds > 0 ? cfg.rounds : (adaptive ? handover_rounds(P) : (parts > 1 ? 16 : 18));
  const int take_below = adaptive ? (cfg.handover_below / parts > 64 ? cfg.handover_below / parts : 64) : 0;
  cudaError_t e = cudaSuccess;
  if (parts > 1) {
    if ((e = cudaEventRecord(ss->fork, stream)) != cudaSuccess) return e;
    for (int p = 1; p < parts; ++p)
      if ((e = cudaStreamWaitEvent(ss->aux[p - 1], ss->fork, 0)) != cudaSuccess) return e;
  }
  const int per = (((B + parts - 1) / parts) + 63) / 64 * 64;
  for (int p = 0; p < parts && e == cudaSuccess; ++p) {
    const int b0 = p * per, b1 = (p + 1) * per < B ? (p + 1) * per : B;
    if (b0 >= b1) continue;
    const CostArgs A = solve_args(B, steps, io, L, desc ? desc + p * kDescInts : nullptr, b0, b1, cfg.warm_start ? cfg.warm_mu : 0.0);
    e = launch_part(P, A, cfg, rounds, take_below, p == 0 ? stream : ss->aux[p - 1], n);
  }
  for (int p = 1; p < parts; ++p) {   // always join, also after an error, so a capture can end cleanly
    cudaError_t e2 = cudaEventRecord(ss->join[p - 1], ss->aux[p - 1]);
    if (e2 == cudaSuccess) e2 = cudaStreamWaitEvent(stream, ss->join[p - 1], 0);
    if (e == cudaSuccess) e = e2;
  }
  return e;
}

// ---------------------------------------------------------------------------------------------
// Pipelined solves on one handle (b200mpc_set_pipeline).  A solve is cut in two launch sequences:
//   bulk  init + rounds in the handle's main workspace; as soon as at most tail.slots problems are still iterating they
//         are moved to the tail context and the main workspace is free for the next batch;
//   tail  rounds (with compaction and the conditional hand-over to the cooperative kernel) + finisher on the tail context.
// The caller orders them with events: bulk(i+1) after bulk(i), tail(i) after bulk(i), bulk(i+depth) after tail(i), so
// the thin tail of one batch -- latency bound: a straggler needs up to hundreds of iterations at long horizons -- runs
// under the bulk of the following batches instead of holding a full-size workspace.  Results do not depend on where a
// problem is finished.
cudaError_t launch_solve_bulk(const Params& P, int B, const SolveIO& io, double* ws, const TailCtx& tail, const SolveConfig& cfg,
                              cudaStream_t stream, long long* n) {
  if (B <= 0) return cudaSuccess;
  const WsLayout L = ws_layout(ws, P.N, B), T = ws_layout(tail.ws, P.N, tail.slots);
  const CostArgs A = solve_args(B, 1, io, L, L.desc, 0, B, 0.0);
  const int rounds = cfg.rounds > 0 ? cfg.rounds : handover_rounds(P);
  mpc_tail_reset_kernel<<<1, 32, 0, stream>>>(T.desc);
  *n += 1;
  launch_init(P, A, stream, n);
  for (int r = 0; r < rounds; ++r) {
    const bool attempt = r + 1 >= cfg.compact_from;
    launch_round(P, A, attempt, stream, n);
    if (attempt) launch_repack(P, A, cfg.compact_max_live, stream, n, tail.slots, T);
  }
  // Whatever never fitted the tail context is finished in place, by the thread loop: in the normal case the workspace
  // is empty by now and the launch must be cheap -- a cooperative-kernel launch, even one that finds nothing to do,
  // asks for 100-200 KB of shared memory per block and has to wait for SMs to drain while the tails of the previous
  // batches keep them busy (measured at N = 100 with 32 tails in flight: ~150 ms per bulk).
  launch_fused(P, A, 0, stream, n);
  return cudaGetLastError();
}

cudaError_t launch_solve_tail(const Params& P, int B, const SolveIO& io, const TailCtx& tail, const SolveConfig& cfg,
                              cudaStream_t stream, long long* n) {
  if (B <= 0) return cudaSuccess;
  const WsLayout L = ws_layout(tail.ws, P.N, tail.slots);
  const CostArgs A = solve_args(B, 1, io, L, L.desc, 0, tail.slots, 0.0);
  // Up to N = 50 the tail is short (the slowest problems need a few dozen iterations): a few rounds, after each of which
  // the cooperative kernel takes the rest over once it fits its resident warps, as in launch_solve.  Above that the tail
  // is long (N = 100: 2 % of the problems need more than 100 iterations, the slowest about 1000) and the tails of many
  // batches are in flight at once: they stay with the compacted thread-per-problem sweeps -- full warps whose blocks come
  // and go, so the tails of all batches share the machine like one large batch -- because the cooperative kernel holds
  // 100 KB of shared memory per problem there (2 resident warps per SM) and a thread loop that runs to completion holds its
  // registers until the slowest problem of the block is done (measured: with either as the finisher of 32 tails in flight
  // the bulk of the following batches runs at a third of its speed).  Only the last few problems go to the cooperative kernel.
  const bool long_tail = P.N > 50;
  const int rounds = long_tail ? 6 * P.N : 10;
  int take_below = 0;
  if (cfg.coop && cfg.handover_below > 0) {
    const int resident = coop_resident_warps(P.N);
    take_below = long_tail ? 32 : (cfg.handover_below < resident ? cfg.handover_below : resident);
    if (take_below > resident) take_below = resident;
    if (take_below > tail.slots) take_below = tail.slots;
  }
  const int coop_every = long_tail ? 8 : 1;
  cudaError_t ce = cudaSuccess;
  for (int r = 0; r < rounds; ++r) {
    launch_round(P, A, true, stream, n);
    launch_repack(P, A, cfg.compact_max_live, stream, n);
    if (take_below > 0 && (r + 1) % coop_every == 0) launch_coop(P, A, 0, take_below, stream, &ce, n);
    if (ce != cudaSuccess) return ce;
  }
  if (take_below > 0) launch_coop(P, A, 0, take_below, stream, &ce, n);
  if (ce != cudaSuccess) return ce;
  // what is left after the last round: the thread loop (the cooperative kernel took over above if the rest fits it)
  launch_fused(P, A, 0, stream, n);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// Adjoint sensitivities of returned solutions (Solver::vjp): one thread per problem, workspace region 0 (slot = problem).
// state6 / coeffs / g_out8 / the gradients (and cost8 / model4, ROWS != kNoRows) in the layout io_aos selects, traj / mult
// / g_traj field-major.  The kModelRows instance also returns grad_model, at the model row or at the handle's values.
template <int ROWS>
using VjpArgsT = typename std::conditional<ROWS != kNoRows, VjpCostIO, VjpIO>::type;
template <int ROWS>
__global__ void __launch_bounds__(kBlock) mpc_vjp_kernel(const __grid_constant__ Params P, const __grid_constant__ VjpArgsT<ROWS> A, double* ws) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= A.B) return;
  const size_t nb = (size_t)A.B, bb = (size_t)b;
  auto at = [&](int k, int n) { return A.io_aos ? bb * n + k : (size_t)k * nb + bb; };   // element k of n of problem b
  Params Q = P;
  Solver<32> S(ROWS ? Q : P, slot_base(P, ws, b), b & 31);
  double s0[6], cf[kMaxCoef], gs6[6], gcf[kMaxCoef], gpar[8];
#pragma unroll
  for (int k = 0; k < 6; ++k) s0[k] = A.state6[at(k, 6)];
#pragma unroll
  for (int i = 0; i < kMaxCoef; ++i) cf[i] = i < A.ncoef ? A.coeffs[at(i, A.ncoef)] : 0.0;
  // an invalid cost or model row: a NaN coefficient makes Solver::vjp return -13 with NaN gradients
  if constexpr (ROWS == kCostRows) {
    if (!cost_row(A.cost8, A.io_aos, A.B, b, Q)) cf[0] = NAN;
  } else if constexpr (ROWS == kModelRows) {
    bool ok = !A.cost8 || cost_row(A.cost8, A.io_aos, A.B, b, Q);
    if (A.model4) ok &= model_row(A.model4, A.io_aos, A.B, b, Q);
    if (!ok) cf[0] = NAN;
  }
  S.set_coeffs(cf, kMaxCoef);
  int st;
  if constexpr (ROWS == kModelRows) {
    double gmod[4];
    st = S.vjp<true>(s0, A.traj + b, nb, A.mult + b, nb, A.g_out8 ? A.g_out8 + at(0, 8) : nullptr, A.io_aos ? 1 : nb,
                     A.g_traj ? A.g_traj + b : nullptr, nb, A.g_obj ? A.g_obj[b] : 0.0, gs6, gcf, gpar, gmod);
    if (A.grad_model)
#pragma unroll
      for (int i = 0; i < 4; ++i) A.grad_model[at(i, 4)] = gmod[i];
  } else {
    st = S.vjp(s0, A.traj + b, nb, A.mult + b, nb, A.g_out8 ? A.g_out8 + at(0, 8) : nullptr, A.io_aos ? 1 : nb,
               A.g_traj ? A.g_traj + b : nullptr, nb, A.g_obj ? A.g_obj[b] : 0.0, gs6, gcf, gpar);
  }
  if (A.grad_state6)
#pragma unroll
    for (int k = 0; k < 6; ++k) A.grad_state6[at(k, 6)] = gs6[k];
  if (A.grad_coeffs)
#pragma unroll
    for (int i = 0; i < kMaxCoef; ++i)
      if (i < A.ncoef) A.grad_coeffs[at(i, A.ncoef)] = gcf[i];
  if (A.grad_params)
#pragma unroll
    for (int i = 0; i < 8; ++i) A.grad_params[at(i, 8)] = gpar[i];
  if (A.status) A.status[b] = st;
}
cudaError_t launch_vjp(const Params& P, const VjpCostIO& io, double* ws, cudaStream_t stream) {
  if (io.B <= 0) return cudaSuccess;
  const int grid = (io.B + kBlock - 1) / kBlock;
  if (io.model4 || io.grad_model) mpc_vjp_kernel<kModelRows><<<grid, kBlock, 0, stream>>>(P, io, ws);
  else if (io.cost8) mpc_vjp_kernel<kCostRows><<<grid, kBlock, 0, stream>>>(P, io, ws);
  else mpc_vjp_kernel<kNoRows><<<grid, kBlock, 0, stream>>>(P, io, ws);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// FP64 peak: 8 independent dependent-FMA chains per thread.
__global__ void __launch_bounds__(256) fp64_peak_kernel(double* sink, int iters) {
  double a0 = threadIdx.x * 1e-3, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
  const double m = 1.0000001, c = 1e-9;
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
      a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
    }
  }
  const double s = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
  if (s == 123.456) sink[0] = s;   // keeps the chains live, never true in practice
}

// ---------------------------------------------------------------------------------------------
// Arithmetic self-test: the sweeps' reciprocal / quotient (drcp / ddiv, mpc_core.cuh) on caller-supplied operands, so a
// test can hold them against the IEEE results.
__global__ void division_selftest_kernel(int n, const double* a, const double* b, double* quot, double* rcp) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  quot[i] = ddiv(a[i], b[i]);
  rcp[i] = drcp(b[i]);
}
cudaError_t launch_division_selftest(int n, const double* a, const double* b, double* quot, double* rcp, cudaStream_t stream) {
  if (n <= 0) return cudaSuccess;
  division_selftest_kernel<<<(n + 255) / 256, 256, 0, stream>>>(n, a, b, quot, rcp);
  return cudaGetLastError();
}

cudaError_t launch_fp64_peak(double* sink, int blocks, int threads, int iters, cudaStream_t stream, double* flop) {
  fp64_peak_kernel<<<blocks, threads, 0, stream>>>(sink, iters);
  *flop = 2.0 * 64.0 * (double)iters * (double)blocks * (double)threads;
  return cudaGetLastError();
}

}  // namespace b200mpc
