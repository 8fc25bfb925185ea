"""udacitympc_b200 -- Python host side of libb200mpc.so, the B200-native drop-in for the mpc_to_line hot path of
cyscgzx33/UdacityMPC.

The interface mirrors the reference's (names, argument meaning, error behaviour):

    reference (C++)                                                 here
    --------------------------------------------------------------  ------------------------------------------
    class MPC { vector<double> Solve(VectorXd x0, VectorXd coeffs) }   MPC().Solve(x0, coeffs)   -> list of 8
      mpc_to_line/src/MPC.h:7-17, solution/MPC.cpp:149-257          MPC().solve_batch(states, coeffs)
    VectorXd polyfit(VectorXd xvals, VectorXd yvals, int order)     polyfit(xvals, yvals, order)
      mpc_to_line/src/helpers.h:24-44                               polyfit_batch(xs, ys, order)
    double polyeval(VectorXd coeffs, double x)  helpers.h:13-19     polyeval(coeffs, x), polyeval_batch(...)
    VectorXd globalKinematic(VectorXd state, VectorXd actuators,    global_kinematic(state, actuators, dt)
      double dt)  global_kinematic_model/solution/main.cpp:36-62    rollout_batch(states, actuators, dt, Lf)

All arithmetic runs in the CUDA library; importing this package without libb200mpc.so (or calling it without a
CUDA device) raises -- there is no CPU fallback.
"""
from .api import (  # noqa: F401
    MODEL_NAMES,
    PARAM_NAMES,
    B200MPCError,
    MPC,
    MPCParams,
    global_kinematic,
    lib_path,
    load_library,
    polyeval,
    polyeval_batch,
    polyfit,
    polyfit_batch,
    read_roadmap_csv,
    roadmap_reference_batch,
    rollout_batch,
    shift_solution,
)

__all__ = ["MODEL_NAMES", "PARAM_NAMES", "B200MPCError", "MPC", "MPCParams", "global_kinematic", "lib_path", "load_library", "polyeval",
           "polyeval_batch", "polyfit", "polyfit_batch", "read_roadmap_csv", "roadmap_reference_batch", "rollout_batch",
           "shift_solution"]
