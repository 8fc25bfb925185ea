/* b200mpc -- C ABI of the B200-native batched nonlinear-MPC solver (libb200mpc.so).
 *
 * This is the drop-in boundary for the reference's mpc_to_line hot path.  Every entry point cites the
 * reference interface it replaces (paths relative to the reference checkout, cyscgzx33/UdacityMPC):
 *
 *   b200mpc_solve_batch        class MPC { std::vector<double> Solve(const VectorXd& x0, const VectorXd& coeffs); }
 *                              mpc_to_line/src/MPC.h:7-17, implementation mpc_to_line/solution/MPC.cpp:149-257
 *                              (FG_eval :45-140; CppAD::ipopt::solve :241-243)
 *   b200mpc_polyfit_batch      VectorXd polyfit(const VectorXd& xvals, const VectorXd& yvals, int order)
 *                              mpc_to_line/src/helpers.h:24-44
 *   b200mpc_polyeval_batch     double polyeval(const VectorXd& coeffs, double x)     mpc_to_line/src/helpers.h:13-19
 *   b200mpc_rollout_batch      VectorXd globalKinematic(const VectorXd& state, const VectorXd& actuators, double dt)
 *                              global_kinematic_model/solution/main.cpp:18-19, 36-62
 *   b200mpc_closed_loop_batch  the feed-forward loop of mpc_to_line/solution/main.cpp:51-76
 *   b200mpc_roadmap_reference_batch  nearest centre-line point + local-frame fit: the producer of (coeffs, cte, epsi)
 *                              that mpc_to_line/src/custom_MPC.cpp:177-212 attempts (solution/main.cpp:25-37 for a line)
 *   b200mpc_params             the file-scope globals of MPC.cpp:14-31 (N, dt, Lf, ref_v), the unit cost weights of
 *                              :57-76, the actuator bounds of :194-203, and the Ipopt options tol / max_iter that
 *                              the option string at :232-235 leaves at their defaults
 *
 * Conventions
 *   - plain pointers and sizes only; no exceptions cross this boundary; every function returns 0 on success or a
 *     negative b200mpc_error, and b200mpc_last_error() describes the most recent failure of the calling thread.
 *   - *_batch functions take HOST buffers in the reference's per-problem ("array of structures") order and do the
 *     host<->device copies themselves; *_batch_device functions take DEVICE buffers in the structure-of-arrays
 *     layout the kernels consume (field-major: element k of problem b at ptr[k*B + b]) and are asynchronous on
 *     the given cudaStream_t (passed as void*; NULL = the handle's own stream).
 *   - a handle is bound to one CUDA device and is the unit of thread safety: one handle per host thread AND one solve
 *     in flight per handle (every call on a handle uses the handle's one workspace and its auxiliary streams; a second
 *     *_device call on the same handle, on whatever stream, first waits on the device for the previous one).
 *   - there is no CPU fallback: without a CUDA device b200mpc_create fails with B200MPC_ERR_CUDA.
 *   - per-problem status values are Ipopt's ApplicationReturnStatus numbers
 *     (Ipopt-3.12.7/Ipopt/src/Interfaces/IpReturnCodes_inc.h:16-39): 0 Solve_Succeeded, 1 Solved_To_Acceptable_Level,
 *     3 Search_Direction_Becomes_Too_Small, 4 Diverging_Iterates, -1 Maximum_Iterations_Exceeded,
 *     -2 Restoration_Failed (the line search failed at an almost feasible point, or b200mpc_set_restoration mode 0),
 *     -3 Error_In_Step_Computation, -13 Invalid_Number_Detected (NaN / Inf in the inputs).  Like MPC::Solve (MPC.cpp:248-249) the solution is returned regardless.
 */
#ifndef B200MPC_H
#define B200MPC_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct b200mpc_params {
  int N;            /* horizon length, MPC.cpp:14 (25) */
  double dt;        /* MPC.cpp:15 (0.05) */
  double Lf;        /* MPC.cpp:27 (2.67) */
  double ref_v;     /* MPC.cpp:31 (40) */
  double w_cte, w_epsi, w_v;     /* MPC.cpp:60-64 (1,1,1) */
  double w_delta, w_a;           /* MPC.cpp:67-70 (1,1) */
  double w_ddelta, w_da;         /* MPC.cpp:73-76 (1,1) */
  double delta_max; /* MPC.cpp:194-195 (0.436332, the literal) */
  double a_max;     /* MPC.cpp:200-201 (1.0) */
  double tol;       /* Ipopt "tol" default 1e-8 */
  int max_iter;     /* Ipopt "max_iter" default 3000 */
} b200mpc_params;

typedef struct b200mpc_handle b200mpc_handle;

enum b200mpc_error {
  B200MPC_OK = 0,
  B200MPC_ERR_ARG = -1,     /* bad argument (null pointer, size out of range, unsupported degree) */
  B200MPC_ERR_CUDA = -2,    /* CUDA runtime error, or no CUDA device */
  B200MPC_ERR_NOMEM = -3    /* device or host allocation failed */
};

#define B200MPC_MAX_COEFFS 4      /* reference polynomial degree <= 3 in the solver */
#define B200MPC_MAX_FIT_POINTS 16 /* polyfit: m <= 16, 1 <= order <= min(m-1, 7) */
#define B200MPC_MAX_FIT_ORDER 7

/* Fills *p with the values the reference hard-codes (see b200mpc_params). */
void b200mpc_default_params(b200mpc_params* p);

/* Creates a solver bound to CUDA device `device`.  Work buffers grow on demand. */
int b200mpc_create(const b200mpc_params* p, int device, b200mpc_handle** out);
void b200mpc_destroy(b200mpc_handle* h);
const char* b200mpc_last_error(void);
/* 8N-2: length of the full variable vector [x|y|psi|v|cte|epsi|delta|a] (MPC.cpp:36-43, 161). */
int b200mpc_num_vars(const b200mpc_handle* h);

/* B independent MPC::Solve calls.
 *   state6  B x 6   (x, y, psi, v, cte, epsi) per problem                 MPC.cpp:152-157
 *   coeffs  B x ncoef, ascending powers, 2 <= ncoef <= 4                  MPC.cpp:117-118 (degree 1 as shipped)
 *   out8    B x 8   (x1, y1, psi1, v1, cte1, epsi1, delta0, a0)           MPC.cpp:253-256
 *   traj    B x (8N-2) full solution in the reference's variable order, or NULL
 *   obj     B       objective value (the "Cost" line, MPC.cpp:251-252), or NULL
 *   status  B       see above, or NULL;   iters  B  interior-point iterations, or NULL */
int b200mpc_solve_batch(b200mpc_handle* h, int B, const double* state6, const double* coeffs, int ncoef, double* out8,
                        double* traj, double* obj, int* status, int* iters);

/* b200mpc_solve_batch without the final wait: the copies in, the solve and the copies out are queued on the handle's own
 * stream and the call returns (truly asynchronous only with pinned host buffers).  The input buffers must stay valid
 * and the output buffers untouched until b200mpc_wait(h) -- which waits for everything queued on the handle -- or a
 * later blocking call on the handle returns.  Lets one host thread keep several handles busy. */
int b200mpc_solve_batch_async(b200mpc_handle* h, int B, const double* state6, const double* coeffs, int ncoef,
                              double* out8, double* traj, double* obj, int* status, int* iters);
int b200mpc_wait(b200mpc_handle* h);

/* Same on device buffers, field-major: d_state6[k*B+b], d_coeffs[i*B+b], d_out8[k*B+b], d_traj[i*B+b]. */
int b200mpc_solve_batch_device(b200mpc_handle* h, int B, const double* d_state6, const double* d_coeffs, int ncoef,
                               double* d_out8, double* d_traj, double* d_obj, int* d_status, int* d_iters,
                               void* stream);

/* The same batch sharded by contiguous index ranges over several handles (normally one per device; several handles on
 * one device are allowed), no inter-device communication (SURVEY 8e): handle g solves
 * problems [g * (B / n), (g + 1) * (B / n)), the last one also the remainder.  Shard 0 is queued and waited for by the
 * calling thread, every other shard by a persistent host thread of the library (created on first use), so the devices
 * start together; one multi call at a time uses those threads (concurrent multi calls are serialised).  Host buffers as
 * b200mpc_solve_batch; pinned ones (cudaHostAlloc / cudaHostRegister) keep the copies asynchronous.
 * Every handle must have been created with the same b200mpc_params and the same restoration mode, and no handle may
 * appear twice (B200MPC_ERR_ARG otherwise: the result rows of the shards would not line up, or two shards would share
 * one workspace). */
int b200mpc_solve_batch_multi(b200mpc_handle* const* hs, int n_handles, int B, const double* state6,
                              const double* coeffs, int ncoef, double* out8, double* traj, double* obj, int* status,
                              int* iters);

/* Closed loop of solution/main.cpp:51-76 for B vehicles: `steps` consecutive solves, each fed the previous solve's
 * predicted state out8[0..5]; the state never leaves the device between steps.
 *   state6  B x 6 initial states, coeffs B x ncoef (constant over the loop)
 *   hist8   steps x B x 8 the returned vector of every step;  cost  steps x B (or NULL);  iters steps x B (or NULL) */
int b200mpc_closed_loop_batch(b200mpc_handle* h, int B, int steps, const double* state6, const double* coeffs,
                              int ncoef, double* hist8, double* cost, int* iters);

/* 10N-4: length of the multiplier vector of one problem, in the reference's order: lambda of the constraint rows
 * x_start+t .. epsi_start+t (6N, MPC.cpp:36-43, 120-138), then z_L of delta_t and a_t (2(N-1)), then z_U of delta_t and
 * a_t (2(N-1)).  The states have no bounds in the reference (+-1e19, MPC.cpp:181-186), so they have no z. */
int b200mpc_num_mults(const b200mpc_handle* h);

/* b200mpc_solve_batch started from a caller-supplied primal-dual point, returning the multipliers.  NOT reference
 * behaviour: the reference cold-starts every call (MPC.cpp:167-177) and reads only x and obj_value from the
 * CppAD::ipopt::solve_result it receives (MPC.cpp:241-256); this is Ipopt's warm_start_init_point
 * (IpWarmStartIterateInitializer) plus the lambda / zl / zu of that solve_result.  The use is a receding-horizon loop
 * that refits the reference every step: start step k+1 from step k's traj and mult shifted by one stage
 * (udacitympc_b200.shift_solution does that).
 *   x_init     B x (8N-2) start point in the layout of traj, or NULL for the default start point.  Its s_0 is replaced by
 *              state6; the controls are pushed 1e-3 max(1, |bound|) inside their bounds.
 *   mult_init  B x (10N-4) multipliers in the layout of mult, or NULL: lambda = 0, z = mu / slack.  Bound multipliers are
 *              kept >= 1e-3.  Needs x_init.
 *   mu_init    initial barrier parameter, in (0, 0.1] (e.g. 1e-4); ignored without x_init
 *   mult       B x (10N-4) the multipliers of the solution, unscaled as Ipopt returns them, or NULL
 * x_init = NULL returns what b200mpc_solve_batch returns, bit for bit, plus mult.  A non-finite entry of a problem's
 * x_init or mult_init gives that problem status -13 (Invalid_Number_Detected), 0 iterations.  The iterations start with
 * a zero-length step that is not counted.  B200MPC_ERR_ARG for mult_init without x_init or mu_init outside (0, 0.1]. */
int b200mpc_solve_batch_warm(b200mpc_handle* h, int B, const double* state6, const double* coeffs, int ncoef,
                             const double* x_init, const double* mult_init, double mu_init, double* out8, double* traj,
                             double* mult, double* obj, int* status, int* iters);
/* Same on device buffers, field-major like b200mpc_solve_batch_device: d_x_init[i*B+b], d_mult_init[i*B+b],
 * d_mult[i*B+b].  Pipelined solves (b200mpc_set_pipeline) accept it like b200mpc_solve_batch_device. */
int b200mpc_solve_batch_warm_device(b200mpc_handle* h, int B, const double* d_state6, const double* d_coeffs, int ncoef,
                                    const double* d_x_init, const double* d_mult_init, double mu_init, double* d_out8,
                                    double* d_traj, double* d_mult, double* d_obj, int* d_status, int* d_iters, void* stream);

/* b200mpc_solve_batch_warm with per-problem cost parameters.  NOT reference behaviour: the reference's cost has one
 * ref_v and one set of weights (MPC.cpp:14-31, 57-76); here a batch of a fleet's vehicles, or of scenes whose weights a
 * network predicts, is solved in one call with each problem's own values.
 *   cost8  B x 8 per problem: ref_v, w_cte, w_epsi, w_v, w_delta, w_a, w_ddelta, w_da (the order of grad_params of
 *          b200mpc_solve_batch_vjp), or NULL for the handle's values (then this is b200mpc_solve_batch_warm).  N, dt, Lf,
 *          the bounds, tol and max_iter stay the handle's.  Weights are not range-checked, like the handle's.
 * A non-finite entry of a problem's cost8 row gives that problem status -13 (Invalid_Number_Detected), 0 iterations.
 * cost8 equal to the handle's values in every row gives what b200mpc_solve_batch_warm gives, bit for bit.  The other
 * arguments and errors are those of b200mpc_solve_batch_warm. */
int b200mpc_solve_batch_cost(b200mpc_handle* h, int B, const double* state6, const double* coeffs, int ncoef, const double* cost8,
                             const double* x_init, const double* mult_init, double mu_init, double* out8, double* traj,
                             double* mult, double* obj, int* status, int* iters);
/* Same on device buffers, field-major like b200mpc_solve_batch_warm_device: d_cost8[k*B+b].  Pipelined solves
 * (b200mpc_set_pipeline) accept it like b200mpc_solve_batch_device. */
int b200mpc_solve_batch_cost_device(b200mpc_handle* h, int B, const double* d_state6, const double* d_coeffs, int ncoef,
                                    const double* d_cost8, const double* d_x_init, const double* d_mult_init, double mu_init,
                                    double* d_out8, double* d_traj, double* d_mult, double* d_obj, int* d_status, int* d_iters,
                                    void* stream);

/* b200mpc_solve_batch_cost with a per-problem vehicle model and actuator limits.  NOT reference behaviour: the reference
 * has one dt, Lf and one pair of bounds (MPC.cpp:14-15, 194-203); here a fleet of vehicles with different wheelbases and
 * steering / acceleration limits is solved in one call, each problem with its own values.
 *   model4  B x 4 per problem: dt, Lf, delta_max, a_max (the fields of b200mpc_params, in that order; the order of
 *           grad_model of b200mpc_solve_batch_vjp_model), or NULL for the handle's values.  N, tol, max_iter and the
 *           restoration mode stay the handle's.
 *   cost8   as in b200mpc_solve_batch_cost, or NULL; either row pointer may be NULL (both NULL: b200mpc_solve_batch_warm).
 * A problem whose model4 row has an entry that is not finite and positive (what b200mpc_create rejects for a handle) gets
 * status -13 (Invalid_Number_Detected) and 0 iterations; the other problems of the batch are unaffected.  model4 equal
 * to the handle's values in every row gives what the call without it gives to the last bits (not bit for bit: the
 * per-problem kernels hold dt, Lf and the bounds in registers, and a few operations round differently there); the same
 * call is bitwise reproducible.  b200mpc_closed_loop_batch and
 * b200mpc_solve_batch_multi do not take per-problem rows.  The other arguments and errors are those of
 * b200mpc_solve_batch_warm. */
int b200mpc_solve_batch_model(b200mpc_handle* h, int B, const double* state6, const double* coeffs, int ncoef, const double* cost8,
                              const double* model4, const double* x_init, const double* mult_init, double mu_init, double* out8,
                              double* traj, double* mult, double* obj, int* status, int* iters);
/* Same on device buffers, field-major like b200mpc_solve_batch_warm_device: d_cost8[k*B+b], d_model4[k*B+b].  Pipelined
 * solves (b200mpc_set_pipeline) accept it like b200mpc_solve_batch_device. */
int b200mpc_solve_batch_model_device(b200mpc_handle* h, int B, const double* d_state6, const double* d_coeffs, int ncoef,
                                     const double* d_cost8, const double* d_model4, const double* d_x_init,
                                     const double* d_mult_init, double mu_init, double* d_out8, double* d_traj, double* d_mult,
                                     double* d_obj, int* d_status, int* d_iters, void* stream);

/* Adjoint sensitivities (vector-Jacobian product) of B solutions: the derivative of a scalar loss L(out8, traj, obj) of
 * each problem's solution w.r.t. its initial state, its reference polynomial and the handle's cost parameters, by the
 * implicit-function theorem at the returned primal-dual point (the differentiable-MPC layer; Ipopt's sIPOPT does the
 * same).  NOT reference behaviour: the reference returns no derivatives.  One Riccati solve of the KKT system of the
 * unscaled problem per problem (about one interior-point iteration), one kernel launch.
 *   state6, coeffs   the inputs of the solve (B x 6, B x ncoef)
 *   traj, mult       B x (8N-2), B x (10N-4): the solution and multipliers b200mpc_solve_batch_warm returned for them.
 *                    They must come from a converged solve (status 0 or 1) on a handle with the same params; the
 *                    derivative is taken at this point as given (its controls are not pushed inside the bounds).
 *   g_out8 (B x 8), g_traj (B x (8N-2)), g_obj (B)   dL/d(out8, traj, obj), or NULL; at least one must be given.
 *                    out8[0..5] is traj's state of t = 1, out8[6], out8[7] its controls of t = 0.
 *   grad_state6 (B x 6), grad_coeffs (B x ncoef), grad_params (B x 8: ref_v, w_cte, w_epsi, w_v, w_delta, w_a, w_ddelta,
 *                    w_da; per problem, a caller sums them), or NULL
 *   status (B) or NULL: 0 ok; -3 a 2x2 control block of the adjoint factorisation is not positive definite at the point
 *                    (not a strict local minimum, or not a point of this handle's problem); -13 a non-finite input.
 *                    The problem's gradients are NaN then.
 * B200MPC_ERR_ARG for a null handle, B <= 0, ncoef outside [2, 4], a null state6 / coeffs / traj / mult or no incoming
 * gradient.  The call uses the handle's workspace and is ordered like a solve on the handle. */
int b200mpc_solve_batch_vjp(b200mpc_handle* h, int B, const double* state6, const double* coeffs, int ncoef, const double* traj,
                            const double* mult, const double* g_out8, const double* g_traj, const double* g_obj,
                            double* grad_state6, double* grad_coeffs, double* grad_params, int* status);
/* Same on device buffers, field-major like b200mpc_solve_batch_warm_device (d_x[i*B+b] for every array), asynchronous
 * on `stream` (NULL: the handle's stream).  Exactly one kernel launch. */
int b200mpc_solve_batch_vjp_device(b200mpc_handle* h, int B, const double* d_state6, const double* d_coeffs, int ncoef,
                                   const double* d_traj, const double* d_mult, const double* d_g_out8, const double* d_g_traj,
                                   const double* d_g_obj, double* d_grad_state6, double* d_grad_coeffs, double* d_grad_params,
                                   int* d_status, void* stream);

/* b200mpc_solve_batch_vjp of solutions of b200mpc_solve_batch_cost: the derivative is taken at each problem's own cost
 * parameters.  NOT reference behaviour.
 *   cost8        B x 8 (ref_v, w_cte, w_epsi, w_v, w_delta, w_a, w_ddelta, w_da) the solve used, or NULL for the handle's
 *                values (then this is b200mpc_solve_batch_vjp)
 *   grad_params  B x 8 in the same order: dL/d(cost8 row) of each problem
 * A non-finite entry of a problem's cost8 row gives that problem status -13 and NaN gradients.  The other arguments and
 * errors are those of b200mpc_solve_batch_vjp. */
int b200mpc_solve_batch_vjp_cost(b200mpc_handle* h, int B, const double* state6, const double* coeffs, int ncoef, const double* cost8,
                                 const double* traj, const double* mult, const double* g_out8, const double* g_traj,
                                 const double* g_obj, double* grad_state6, double* grad_coeffs, double* grad_params, int* status);
/* Same on device buffers, field-major like b200mpc_solve_batch_vjp_device: d_cost8[k*B+b].  Exactly one kernel launch. */
int b200mpc_solve_batch_vjp_cost_device(b200mpc_handle* h, int B, const double* d_state6, const double* d_coeffs, int ncoef,
                                        const double* d_cost8, const double* d_traj, const double* d_mult, const double* d_g_out8,
                                        const double* d_g_traj, const double* d_g_obj, double* d_grad_state6, double* d_grad_coeffs,
                                        double* d_grad_params, int* d_status, void* stream);

/* b200mpc_solve_batch_vjp_cost of solutions of b200mpc_solve_batch_model: the derivative is taken at each problem's own
 * cost and model parameters, and also w.r.t. the model.  NOT reference behaviour.
 *   cost8, model4  the rows the solve used, or NULL for the handle's values (either may be NULL)
 *   grad_model     B x 4 (dt, Lf, delta_max, a_max): dL/d(model4 row) of each problem, or NULL.  With model4 NULL it is
 *                  taken at the handle's values; summed over the batch, that is the gradient w.r.t. the shared model.
 * A problem whose model4 row has an entry that is not finite and positive gets status -13 and NaN gradients.  The other
 * arguments and errors are those of b200mpc_solve_batch_vjp_cost. */
int b200mpc_solve_batch_vjp_model(b200mpc_handle* h, int B, const double* state6, const double* coeffs, int ncoef, const double* cost8,
                                  const double* model4, const double* traj, const double* mult, const double* g_out8,
                                  const double* g_traj, const double* g_obj, double* grad_state6, double* grad_coeffs,
                                  double* grad_params, double* grad_model, int* status);
/* Same on device buffers, field-major like b200mpc_solve_batch_vjp_device: d_model4[k*B+b], d_grad_model[k*B+b].  Exactly
 * one kernel launch. */
int b200mpc_solve_batch_vjp_model_device(b200mpc_handle* h, int B, const double* d_state6, const double* d_coeffs, int ncoef,
                                         const double* d_cost8, const double* d_model4, const double* d_traj, const double* d_mult,
                                         const double* d_g_out8, const double* d_g_traj, const double* d_g_obj,
                                         double* d_grad_state6, double* d_grad_coeffs, double* d_grad_params,
                                         double* d_grad_model, int* d_status, void* stream);

/* Forward sensitivities (Jacobian-vector product) of B solutions: the derivative of each problem's solution (out8, traj,
 * obj) along a tangent of its inputs -- initial state, reference polynomial, cost parameters and vehicle model -- by the
 * implicit-function theorem at the returned primal-dual point: K [dx; dlam] = -dF/dtheta dtheta with the KKT matrix K of
 * b200mpc_solve_batch_vjp (the transpose of that call: <v, J u> from this call equals <J^T v, u> from it up to
 * rounding).  NOT reference behaviour: the reference returns no derivatives.  One Riccati solve of the KKT system of the
 * unscaled problem per problem and tangent, one kernel launch.
 *   state6, coeffs, cost8, model4, traj, mult   as for b200mpc_solve_batch_vjp_model (cost8 / model4 may be NULL: the
 *                    handle's values)
 *   t_state6 (B x 6), t_coeffs (B x ncoef), t_cost8 (B x 8), t_model4 (B x 4)   the tangent, in the orders of state6,
 *                    coeffs, cost8 and model4, or NULL for zero; at least one must be given.  t_model4 with model4 NULL
 *                    is taken at the handle's values.
 *   t_out8 (B x 8), t_traj (B x (8N-2))   d out8, d traj, or NULL.  t_traj's states of t = 0 are t_state6; t_out8 is
 *                    t_traj's state of t = 1 and controls of t = 0.  Controls are not clamped to the bounds as traj's are.
 *   t_obj (B) or NULL   d obj in the envelope form df/dtheta + lambda^T dc/dtheta (bound terms included), the exact
 *                    transpose of g_obj's term of the VJP; it agrees with grad f . dx + df/dtheta to the solver tolerance.
 *   status (B) or NULL: as b200mpc_solve_batch_vjp (a non-finite tangent also gives -13); the outputs are NaN then.
 * B200MPC_ERR_ARG for a null handle, B <= 0, ncoef outside [2, 4], a null state6 / coeffs / traj / mult or no tangent.
 * The call uses the handle's workspace and is ordered like a solve on the handle. */
int b200mpc_solve_batch_jvp(b200mpc_handle* h, int B, const double* state6, const double* coeffs, int ncoef, const double* cost8,
                            const double* model4, const double* traj, const double* mult, const double* t_state6,
                            const double* t_coeffs, const double* t_cost8, const double* t_model4, double* t_out8,
                            double* t_traj, double* t_obj, int* status);
/* Same on device buffers, field-major like b200mpc_solve_batch_vjp_device (d_x[i*B+b] for every array), asynchronous on
 * `stream` (NULL: the handle's stream).  Exactly one kernel launch. */
int b200mpc_solve_batch_jvp_device(b200mpc_handle* h, int B, const double* d_state6, const double* d_coeffs, int ncoef,
                                   const double* d_cost8, const double* d_model4, const double* d_traj, const double* d_mult,
                                   const double* d_t_state6, const double* d_t_coeffs, const double* d_t_cost8,
                                   const double* d_t_model4, double* d_t_out8, double* d_t_traj, double* d_t_obj, int* d_status,
                                   void* stream);

/* Warm start for b200mpc_closed_loop_batch (SURVEY 8f; NOT reference behaviour: the reference cold-starts every call,
 * MPC.cpp:167-177, and so does this library unless enabled here).  When enabled, every step after the first starts from
 * the previous step's solution shifted by one stage, with the barrier parameter at mu_init (e.g. 1e-4).  The optimum
 * reached is the same local optimum within the solver tolerance; the iterates, iteration counts and last digits of
 * weakly active bounds differ from a cold start. */
int b200mpc_set_warm_start(b200mpc_handle* h, int enable, double mu_init);

/* Internal concurrency of one large solve call: the batch is cut into `parts` (1..4) contiguous sub-batches whose
 * kernels run concurrently on internal streams (joined before the call's stream continues, so the call keeps its
 * stream-ordered semantics).  Results do not depend on it for a fixed number of rounds (with the automatic setting of
 * b200mpc_set_solver_mode the hand-over to the cooperative kernel adapts to the sub-batch, which can change the last
 * bit of the few problems that finish on the other side of it).  Default 4: best for a caller that issues one call at a
 * time; a caller that already overlaps several calls on several handles / streams should set 1. */
int b200mpc_set_batch_split(b200mpc_handle* h, int parts);

/* Hand-over of the thin tail of a batch to the cooperative (warp-per-problem) kernel: after every round from
 * `from_round` on, once the batch has been compacted to at most `occupied_slots` problems, that kernel finishes them
 * (0 = only after the last round).  The cooperative kernel advances a problem 6x faster than the sweeps do but costs
 * 12x the machine time per iteration, so the threshold trades the latency of a lone call against the throughput of
 * overlapped calls: default 1184 from round 14 (its resident warps on a B200; best for one call at a time); a caller
 * that overlaps several calls on several handles / streams should set about 64-256 (measured with 64, 65 536 / 8 192
 * problems per call: +2 % / +11 % solves/s; a lone 8 192-problem call gets 13 % slower with 0).  Results do not depend on it beyond the last bits a
 * hand-over may change. */
int b200mpc_set_handover(b200mpc_handle* h, int occupied_slots, int from_round);

/* Pipelined solves on one handle (the generalisation of the one-call-at-a-time loop of solution/main.cpp:51-54 to a
 * stream of batches).  Iteration counts have a thin, long tail (N = 25: mean 12, a few problems in 10^5 need 30-50;
 * N = 100: mean 19, 2 % need more than 100, the slowest about 1000), and a batch is done when its slowest problem is.
 * With depth > 0 every b200mpc_solve_batch_device call of more than tail_slots problems is queued in two parts: the
 * bulk runs in the handle's full-size workspace until at most tail_slots problems are still iterating; those move to one
 * of `depth` small tail contexts (used round robin) and finish there, while the next call's bulk already runs.  Calls
 * stay stream-ordered for their caller -- the outputs of a call are complete when the work queued on ITS stream is --
 * so the overlap exists between calls issued on DIFFERENT streams (the bulks are ordered among themselves by the
 * library).  Memory: depth x the workspace of tail_slots problems instead of one full workspace per overlapped call.
 * Results do not depend on it beyond the last bits a hand-over between the thread-per-problem sweeps and the
 * cooperative kernel may change.  depth = 0 (default) switches it off; it synchronises the device. */
int b200mpc_set_pipeline(b200mpc_handle* h, int depth, int tail_slots);

/* Batch compaction of the throughput path: after every round from `from_round` on, when the problems that are still
 * iterating fill at most `max_live_fraction` of the occupied workspace slots, they are moved to consecutive slots, so
 * the following rounds run full warps on whole memory sectors instead of a few lanes per warp.  Results do not
 * depend on it.  Default 0.7 from round 4; 0 switches it off. */
int b200mpc_set_compaction(b200mpc_handle* h, double max_live_fraction, int from_round);

/* What follows a failed line search (Ipopt: IpBacktrackingLineSearch.cpp:498-585 -> soft restoration phase, then
 * IpRestoMinC_1Nrm.cpp).  Never reached on the benchmark workloads at the reference's N = 25; 1 % of problems with
 * initial states far off the road and 2 % of the problems at N = 100 get there.
 *   mode 0: such a problem returns status -2 (Restoration_Failed) at the iteration where Ipopt would switch.
 *   mode 1: the restoration step -- a forward sweep removes 5 % of every constraint defect with the controls
 *           kept, the point left enters the filter, lambda is reset to 0, z moves towards mu / slack -- i.e. what Ipopt
 *           does around its restoration phase, with a closed-form point instead of Ipopt's nested restoration solve.
 *           NOT a restatement of that solve: the iteration count of such a problem differs from Ipopt's; the solution
 *           is the reference's on 346 / 346 (N = 25), 14 / 14 (N = 50), 170 / 179 (N = 100) such problems (DESIGN.md 3).
 *   mode 2 (default): as 1, preceded by Ipopt's soft restoration phase (damped full primal-dual steps accepted on the primal-dual
 *           system error, IpBacktrackingLineSearch.cpp:1043-1140), restated exactly: the few problems on which Ipopt
 *           takes such steps then keep its iterates and iteration count. */
int b200mpc_set_restoration(b200mpc_handle* h, int mode);

/* B least-squares polynomial fits (unpivoted Householder QR of the Vandermonde matrix, as Eigen 3.3.3 does for
 * helpers.h:24-44).  xs, ys: B x m;  coeffs_out: B x (order+1).  Requires 1 <= order <= m-1 (helpers.h:26 assert). */
int b200mpc_polyfit_batch(b200mpc_handle* h, int B, const double* xs, const double* ys, int m, int order,
                          double* coeffs_out);
/* Device buffers, field-major: d_xs[j*B+b], d_ys[j*B+b], d_coeffs_out[i*B+b]. */
int b200mpc_polyfit_batch_device(b200mpc_handle* h, int B, const double* d_xs, const double* d_ys, int m, int order,
                                 double* d_coeffs_out, void* stream);

/* y[b] = sum_i coeffs[b][i] * x[b]^i  (helpers.h:13-19).  coeffs: B x ncoef, 1 <= ncoef <= 64. */
int b200mpc_polyeval_batch(b200mpc_handle* h, int B, const double* coeffs, int ncoef, const double* x, double* y);
/* Device buffers, field-major: d_coeffs[i*B+b], d_x[b], d_y[b]; 1 <= ncoef <= 64. */
int b200mpc_polyeval_batch_device(b200mpc_handle* h, int B, const double* d_coeffs, int ncoef, const double* d_x,
                                  double* d_y, void* stream);

/* B bicycle-model rollouts of H Euler steps (global_kinematic_model/solution/main.cpp:36-62; H=1 is globalKinematic).
 *   state4 B x 4 (x,y,psi,v);  act B x H x 2 (delta,a);  out B x H x 4 (the state after each step).
 *   1 <= H <= 1024 on this host entry, 1 <= H <= 4096 on the device entry; Lf > 0. */
int b200mpc_rollout_batch(b200mpc_handle* h, int B, int H, const double* state4, const double* act, double dt,
                          double Lf, double* out);
/* Device buffers, field-major: d_state4[k*B+b], d_act[(s*2+j)*B+b], d_out[(s*4+k)*B+b]. */
int b200mpc_rollout_batch_device(b200mpc_handle* h, int B, int H, const double* d_state4, const double* d_act,
                                 double dt, double Lf, double* d_out, void* stream);

/* Roadmap front-end (the step in front of MPC::Solve; SURVEY 8f): for B vehicle poses in the road's global frame,
 * nearest centre-line point (what mpc_to_line/src/custom_MPC.cpp:177-185 computes), the 6 consecutive centre-line
 * points from there, global -> vehicle frame, degree-3 polyfit, and the MPC inputs in the vehicle frame:
 * state6 = (0, 0, 0, v, cte = p(0), epsi = -atan(p'(0))) as solution/main.cpp:34-37 defines cte / epsi.
 *   pose4  B x 4 (x, y, psi, v);  centerline  n_wp x 2 (x, y), 6 <= n_wp <= 12000 (e.g. columns 4,5 of mpc_to_line/roadmap.csv)
 *   state6_out  B x 6;  coeffs_out  B x 4 -- ready for b200mpc_solve_batch(..., ncoef = 4, ...) */
int b200mpc_roadmap_reference_batch(b200mpc_handle* h, int B, const double* pose4, const double* centerline, int n_wp,
                                    double* state6_out, double* coeffs_out);
/* Device buffers: d_pose4[k*B+b] (field-major), d_centerline[i*2+j] (row-major), d_state6_out[k*B+b], d_coeffs_out[i*B+b]. */
int b200mpc_roadmap_reference_batch_device(b200mpc_handle* h, int B, const double* d_pose4, const double* d_centerline,
                                           int n_wp, double* d_state6_out, double* d_coeffs_out, void* stream);

/* Reads a roadmap file in the reference's format (mpc_to_line/roadmap.csv: 7 comma-separated numbers per line -- left
 * edge x, y, right edge x, y, centre line x, y, slope) the way CustomMPC::readRoadmapFromCSV / parseRoadMapLine intend to
 * (mpc_to_line/src/custom_MPC.h:25-44; the constructor at custom_MPC.cpp:201-212 keeps columns 4, 5 as the centre line
 * and atan(column 6) as its direction): one waypoint per line, fields split at ','.  The reference converts every field
 * with std::stof, i.e. through SINGLE precision; float_fields != 0 reproduces that, 0 parses doubles.  Host-only (no
 * device, no handle).  The reference's reader opens the file NAME as a string stream (custom_MPC.h:28) and so never
 * reads the file; that bug is not reproduced.
 *   centerline_out  max_wp x 2, or NULL;  slope_out  max_wp, or NULL;  *n_wp = waypoints in the file (may exceed
 *   max_wp: only the first max_wp are written) -- feed centerline_out to b200mpc_roadmap_reference_batch. */
int b200mpc_read_roadmap_csv(const char* path, int float_fields, double* centerline_out, double* slope_out, int max_wp, int* n_wp);

/* Execution mode of the solver (tuning; results do not depend on it).
 *   mode 0 (default)  throughput path + latency path.  Batches of at least `fused_below` problems (default 3072) run
 *                     rounds of the per-pass thread-per-problem kernels (factor, forward, step).  By default the
 *                     number of rounds adapts to the batch: after every round from the 14th on (at most 20) the
 *                     cooperative kernel takes the rest over as soon as the compacted batch fits one of its waves
 *                     (1184 problems); a positive `rounds` fixes the hand-over point instead;
 *                     whatever is still iterating then -- the thin tail of the batch and rare 30-50 iteration
 *                     stragglers -- is finished by the cooperative warp-per-problem kernel.  Smaller batches (e.g. the
 *                     reference's one-problem MPC::Solve call: 0.6 ms) use the cooperative kernel alone.
 *   mode 1            the fused thread-per-problem kernel alone (one launch per solve; kept for comparison)
 * rounds <= 0 / fused_below < 0 keep the current value.  The whole launch sequence of a solve is replayed as one CUDA graph. */
int b200mpc_set_solver_mode(b200mpc_handle* h, int mode, int rounds, int fused_below);

/* Measurement helpers (used by bench.py; not part of the reference interface). */
/* Off by default.  When enabled, every solve is bracketed by a pair of CUDA events on its stream (kept until
 * b200mpc_kernel_time_ms reads / resets them; at most 8192 pairs). */
int b200mpc_set_timing(b200mpc_handle* h, int enable);
/* Total device time in ms of the solver's kernels (one interval per batch: first to last kernel of a solve) since the
 * last reset, measured with CUDA events on the launching stream, and the number of intervals (0 with timing off). */
int b200mpc_kernel_time_ms(b200mpc_handle* h, double* total_ms, int* launches, int reset);
/* Sustained FP64 FMA throughput of the device in TFLOP/s (dependent-chain DFMA microbenchmark, 2 FLOP per FMA). */
int b200mpc_measure_fp64_peak(b200mpc_handle* h, double* tflops);
/* Arithmetic self-test (host arrays of n doubles): quot[i] = a[i] / b[i] and rcp[i] = 1 / b[i] as the sweeps compute
 * them -- rcp.approx.ftz.f64 refined by Newton steps, within 1 ulp of the IEEE result for operands in the normal range,
 * +-inf / 0 / NaN like the exact operation for a zero or infinite divisor -- so a caller (tests/test_gpu_parity.py) can
 * hold the library's arithmetic against its own.  No reference counterpart: Ipopt divides with the host FPU. */
int b200mpc_selftest_division(b200mpc_handle* h, int n, const double* a, const double* b, double* quot, double* rcp);
/* Number of kernels this handle has launched since creation. */
long long b200mpc_launch_count(const b200mpc_handle* h);

#ifdef __cplusplus
}
#endif
#endif /* B200MPC_H */
