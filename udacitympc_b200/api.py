"""ctypes binding of include/b200mpc.h and the reference-shaped Python wrappers around it."""
import ctypes
import os
import threading

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
_dp = ctypes.POINTER(ctypes.c_double)
_ip = ctypes.POINTER(ctypes.c_int)
_vp = ctypes.c_void_p


class B200MPCError(RuntimeError):
    pass


class MPCParams(ctypes.Structure):
    """b200mpc_params: the reference's hard-coded configuration (MPC.cpp:14-31, 57-76, 194-203) + Ipopt tol/max_iter."""
    _fields_ = [("N", ctypes.c_int), ("dt", ctypes.c_double), ("Lf", ctypes.c_double), ("ref_v", ctypes.c_double),
                ("w_cte", ctypes.c_double), ("w_epsi", ctypes.c_double), ("w_v", ctypes.c_double),
                ("w_delta", ctypes.c_double), ("w_a", ctypes.c_double), ("w_ddelta", ctypes.c_double),
                ("w_da", ctypes.c_double), ("delta_max", ctypes.c_double), ("a_max", ctypes.c_double),
                ("tol", ctypes.c_double), ("max_iter", ctypes.c_int)]


# every symbol include/b200mpc.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "b200mpc_default_params": (None, [ctypes.POINTER(MPCParams)]),
    "b200mpc_create": (ctypes.c_int, [ctypes.POINTER(MPCParams), ctypes.c_int, ctypes.POINTER(_vp)]),
    "b200mpc_destroy": (None, [_vp]),
    "b200mpc_last_error": (ctypes.c_char_p, []),
    "b200mpc_num_vars": (ctypes.c_int, [_vp]),
    "b200mpc_num_mults": (ctypes.c_int, [_vp]),
    "b200mpc_solve_batch": (ctypes.c_int, [_vp, ctypes.c_int, _dp, _dp, ctypes.c_int, _dp, _dp, _dp, _ip, _ip]),
    "b200mpc_solve_batch_async": (ctypes.c_int, [_vp, ctypes.c_int, _dp, _dp, ctypes.c_int, _dp, _dp, _dp, _ip, _ip]),
    "b200mpc_wait": (ctypes.c_int, [_vp]),
    "b200mpc_solve_batch_device": (ctypes.c_int, [_vp, ctypes.c_int, _vp, _vp, ctypes.c_int, _vp, _vp, _vp, _vp, _vp, _vp]),
    "b200mpc_solve_batch_warm": (ctypes.c_int, [_vp, ctypes.c_int, _dp, _dp, ctypes.c_int, _dp, _dp, ctypes.c_double, _dp, _dp,
                                                _dp, _dp, _ip, _ip]),
    "b200mpc_solve_batch_warm_device": (ctypes.c_int, [_vp, ctypes.c_int, _vp, _vp, ctypes.c_int, _vp, _vp, ctypes.c_double, _vp,
                                                       _vp, _vp, _vp, _vp, _vp, _vp]),
    "b200mpc_solve_batch_cost": (ctypes.c_int, [_vp, ctypes.c_int, _dp, _dp, ctypes.c_int, _dp, _dp, _dp, ctypes.c_double, _dp,
                                                _dp, _dp, _dp, _ip, _ip]),
    "b200mpc_solve_batch_cost_device": (ctypes.c_int, [_vp, ctypes.c_int, _vp, _vp, ctypes.c_int, _vp, _vp, _vp, ctypes.c_double,
                                                       _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "b200mpc_solve_batch_vjp_cost": (ctypes.c_int, [_vp, ctypes.c_int, _dp, _dp, ctypes.c_int] + [_dp] * 9 + [_ip]),
    "b200mpc_solve_batch_vjp_cost_device": (ctypes.c_int, [_vp, ctypes.c_int, _vp, _vp, ctypes.c_int] + [_vp] * 11),
    "b200mpc_solve_batch_model": (ctypes.c_int, [_vp, ctypes.c_int, _dp, _dp, ctypes.c_int, _dp, _dp, _dp, _dp, ctypes.c_double,
                                                 _dp, _dp, _dp, _dp, _ip, _ip]),
    "b200mpc_solve_batch_model_device": (ctypes.c_int, [_vp, ctypes.c_int, _vp, _vp, ctypes.c_int, _vp, _vp, _vp, _vp,
                                                        ctypes.c_double, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "b200mpc_solve_batch_vjp_model": (ctypes.c_int, [_vp, ctypes.c_int, _dp, _dp, ctypes.c_int] + [_dp] * 11 + [_ip]),
    "b200mpc_solve_batch_vjp_model_device": (ctypes.c_int, [_vp, ctypes.c_int, _vp, _vp, ctypes.c_int] + [_vp] * 13),
    "b200mpc_solve_batch_vjp": (ctypes.c_int, [_vp, ctypes.c_int, _dp, _dp, ctypes.c_int, _dp, _dp, _dp, _dp, _dp, _dp, _dp, _dp,
                                               _ip]),
    "b200mpc_solve_batch_vjp_device": (ctypes.c_int, [_vp, ctypes.c_int, _vp, _vp, ctypes.c_int] + [_vp] * 10),
    "b200mpc_solve_batch_jvp": (ctypes.c_int, [_vp, ctypes.c_int, _dp, _dp, ctypes.c_int] + [_dp] * 11 + [_ip]),
    "b200mpc_solve_batch_jvp_device": (ctypes.c_int, [_vp, ctypes.c_int, _vp, _vp, ctypes.c_int] + [_vp] * 13),
    "b200mpc_solve_batch_multi": (ctypes.c_int, [ctypes.POINTER(_vp), ctypes.c_int, ctypes.c_int, _dp, _dp, ctypes.c_int,
                                                 _dp, _dp, _dp, _ip, _ip]),
    "b200mpc_closed_loop_batch": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, _dp, _dp, ctypes.c_int, _dp, _dp, _ip]),
    "b200mpc_polyfit_batch": (ctypes.c_int, [_vp, ctypes.c_int, _dp, _dp, ctypes.c_int, ctypes.c_int, _dp]),
    "b200mpc_polyfit_batch_device": (ctypes.c_int, [_vp, ctypes.c_int, _vp, _vp, ctypes.c_int, ctypes.c_int, _vp, _vp]),
    "b200mpc_polyeval_batch": (ctypes.c_int, [_vp, ctypes.c_int, _dp, ctypes.c_int, _dp, _dp]),
    "b200mpc_polyeval_batch_device": (ctypes.c_int, [_vp, ctypes.c_int, _vp, ctypes.c_int, _vp, _vp, _vp]),
    "b200mpc_rollout_batch": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, _dp, _dp, ctypes.c_double, ctypes.c_double, _dp]),
    "b200mpc_rollout_batch_device": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, _vp, _vp, ctypes.c_double,
                                                    ctypes.c_double, _vp, _vp]),
    "b200mpc_roadmap_reference_batch": (ctypes.c_int, [_vp, ctypes.c_int, _dp, _dp, ctypes.c_int, _dp, _dp]),
    "b200mpc_roadmap_reference_batch_device": (ctypes.c_int, [_vp, ctypes.c_int, _vp, _vp, ctypes.c_int, _vp, _vp, _vp]),
    "b200mpc_read_roadmap_csv": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_int, _dp, _dp, ctypes.c_int, _ip]),
    "b200mpc_set_warm_start": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_double]),
    "b200mpc_set_batch_split": (ctypes.c_int, [_vp, ctypes.c_int]),
    "b200mpc_set_compaction": (ctypes.c_int, [_vp, ctypes.c_double, ctypes.c_int]),
    "b200mpc_set_pipeline": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int]),
    "b200mpc_set_handover": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int]),
    "b200mpc_set_restoration": (ctypes.c_int, [_vp, ctypes.c_int]),
    "b200mpc_set_solver_mode": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    "b200mpc_set_timing": (ctypes.c_int, [_vp, ctypes.c_int]),
    "b200mpc_kernel_time_ms": (ctypes.c_int, [_vp, _dp, _ip, ctypes.c_int]),
    "b200mpc_measure_fp64_peak": (ctypes.c_int, [_vp, _dp]),
    "b200mpc_selftest_division": (ctypes.c_int, [_vp, ctypes.c_int, _dp, _dp, _dp, _dp]),
    "b200mpc_launch_count": (ctypes.c_longlong, [_vp]),
}

_lib = None
_lib_lock = threading.Lock()


def lib_path():
    """In-tree library; B200MPC_LIB selects another build of the same library (kernel tuning experiments)."""
    return os.environ.get("B200MPC_LIB") or os.path.join(_PKG, "lib", "libb200mpc.so")


def load_library():
    """Loads libb200mpc.so (built in-tree by udacitympc_b200.build).  Raises if it is missing: no fallback."""
    global _lib
    with _lib_lock:
        if _lib is None:
            path = lib_path()
            if not os.path.exists(path):
                raise B200MPCError(
                    f"{path} not found: build it with `python -m udacitympc_b200.build` "
                    "(the CUDA library is the only compute path; there is no CPU fallback)")
            L = ctypes.CDLL(path)
            for name, (res, args) in SYMBOLS.items():
                fn = getattr(L, name)   # AttributeError if the library does not export a declared symbol
                fn.restype = res
                fn.argtypes = args
            _lib = L
    return _lib


def _check(rc):
    if rc != 0:
        raise B200MPCError(f"b200mpc error {rc}: {load_library().b200mpc_last_error().decode()}")


def _f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None:
        a = a.reshape(shape)
    return a


def _ptr(a):
    return a.ctypes.data_as(_dp)


def default_params(**kw):
    p = MPCParams()
    load_library().b200mpc_default_params(ctypes.byref(p))
    for k, v in kw.items():
        if not hasattr(p, k):
            raise TypeError(f"unknown parameter {k}")
        setattr(p, k, v)
    return p


# the parameters b200mpc_solve_batch_vjp differentiates, in the order of its grad_params (and of a cost8 row)
PARAM_NAMES = ("ref_v", "w_cte", "w_epsi", "w_v", "w_delta", "w_a", "w_ddelta", "w_da")


def _cost8(cost_params, B):
    """(B, 8) or (8,) broadcast, in PARAM_NAMES order -> the (B, 8) float64 rows b200mpc_solve_batch_cost takes."""
    c = _f64(cost_params)
    if c.ndim == 1:
        c = np.broadcast_to(c, (B, c.size))
    if c.shape != (B, 8):
        raise ValueError(f"cost_params must be (B, 8) or (8,) in the order {PARAM_NAMES}")
    return np.ascontiguousarray(c)


# the vehicle model parameters of a model4 row, in the order of b200mpc_params (and of grad_model)
MODEL_NAMES = ("dt", "Lf", "delta_max", "a_max")


def _model4(model_params, B):
    """(B, 4) or (4,) broadcast, in MODEL_NAMES order -> the (B, 4) float64 rows b200mpc_solve_batch_model takes."""
    c = _f64(model_params)
    if c.ndim == 1:
        c = np.broadcast_to(c, (B, c.size))
    if c.shape != (B, 4):
        raise ValueError(f"model_params must be (B, 4) or (4,) in the order {MODEL_NAMES}")
    return np.ascontiguousarray(c)


class MPC:
    """Drop-in for the reference's `class MPC` (mpc_to_line/src/MPC.h:7-17).

    `MPC().Solve(x0, coeffs)` returns `[x1, y1, psi1, v1, cte1, epsi1, delta0, a0]` exactly like
    solution/MPC.cpp:253-256.  Unlike the reference the configuration is not a set of edit-the-source globals
    (MPC.cpp:14-31) but keyword parameters with the same defaults, and batches are first class.
    Like the reference, Solve ignores the solver status (MPC.cpp:248-249); `last_status` exposes it."""

    def __init__(self, device=0, print_cost=False, full_polynomial=False, **params):
        self._lib = load_library()
        self.params = default_params(**params)
        self.device = device
        self.print_cost = print_cost
        # Solve(): the reference's FG_eval reads coeffs[0..1] only (MPC.cpp:117-118) whatever the vector's length, and
        # so does Solve() unless this extension is switched on (solve_batch always uses every column it is given)
        self.full_polynomial = full_polynomial
        h = _vp()
        _check(self._lib.b200mpc_create(ctypes.byref(self.params), device, ctypes.byref(h)))
        self._h = h
        self.last_status = None
        self.last_iters = None
        self.last_cost = None

    # -- lifetime
    def close(self):
        if getattr(self, "_h", None):
            self._lib.b200mpc_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    @property
    def handle(self):
        return self._h

    @property
    def num_vars(self):
        return self._lib.b200mpc_num_vars(self._h)

    @property
    def num_mults(self):
        """10N-4: lambda of the 6N constraint rows, then z_L and z_U of the 2(N-1) controls (b200mpc_num_mults)."""
        return self._lib.b200mpc_num_mults(self._h)

    # -- the reference call
    def Solve(self, x0, coeffs):
        x0 = _f64(x0).ravel()
        coeffs = _f64(coeffs).ravel()
        if x0.size != 6:
            raise ValueError("state must have 6 entries (x, y, psi, v, cte, epsi)")
        if coeffs.size < 2:
            raise ValueError("coeffs must have at least 2 entries (MPC.cpp:117-118)")
        if not self.full_polynomial:
            coeffs = coeffs[:2]
        r = self.solve_batch(x0[None, :], coeffs[None, :], want_traj=False)
        self.last_status = int(r["status"][0])
        self.last_iters = int(r["iters"][0])
        self.last_cost = float(r["cost"][0])
        if self.print_cost:
            print(f"Cost {self.last_cost:g}")   # MPC.cpp:251-252
        return [float(v) for v in r["out8"][0]]

    # -- batched host-buffer call
    def solve_batch(self, states, coeffs, want_traj=False, x_init=None, mult_init=None, mu_init=1e-4, want_mult=False,
                    cost_params=None, model_params=None):
        """states (B,6), coeffs (B,ncoef) or (ncoef,) shared by all problems.  Returns dict(out8 (B,8), cost (B,),
        status (B,), iters (B,), traj (B,8N-2) if requested, mult (B,10N-4) if requested).

        Warm start (not reference behaviour, b200mpc_solve_batch_warm): x_init (B,8N-2) in the layout of traj and
        optionally mult_init (B,10N-4) in the layout of mult start the solve there with the barrier parameter mu_init;
        shift_solution() turns one receding-horizon step's traj / mult into the next step's start.

        Per-problem costs (not reference behaviour, b200mpc_solve_batch_cost): cost_params (B,8) or (8,) shared, in the
        order PARAM_NAMES, replaces the handle's ref_v and weights problem by problem; None uses the handle's.

        Per-problem vehicles (not reference behaviour, b200mpc_solve_batch_model): model_params (B,4) or (4,) shared, in
        the order MODEL_NAMES, replaces the handle's dt, Lf, delta_max and a_max problem by problem; None uses the
        handle's."""
        states = _f64(states)
        if states.ndim != 2 or states.shape[1] != 6:
            raise ValueError("states must be (B, 6)")
        B = states.shape[0]
        coeffs = _f64(coeffs)
        if coeffs.ndim == 1:
            coeffs = np.ascontiguousarray(np.broadcast_to(coeffs, (B, coeffs.size)))
        if coeffs.shape[0] != B:
            raise ValueError("coeffs must be (B, ncoef)")
        ncoef = coeffs.shape[1]
        out8 = np.empty((B, 8))
        cost = np.empty(B)
        status = np.empty(B, dtype=np.int32)
        iters = np.empty(B, dtype=np.int32)
        traj = np.empty((B, self.num_vars)) if want_traj else None
        if model_params is not None:
            m4 = _model4(model_params, B)
            c8 = None if cost_params is None else _cost8(cost_params, B)
            x_init = None if x_init is None else _f64(x_init, (B, self.num_vars))
            mult_init = None if mult_init is None else _f64(mult_init, (B, self.num_mults))
            mult = np.empty((B, self.num_mults)) if want_mult else None
            _check(self._lib.b200mpc_solve_batch_model(
                self._h, B, _ptr(states), _ptr(coeffs), ncoef, None if c8 is None else _ptr(c8), _ptr(m4),
                None if x_init is None else _ptr(x_init), None if mult_init is None else _ptr(mult_init), float(mu_init),
                _ptr(out8), _ptr(traj) if want_traj else None, _ptr(mult) if want_mult else None, _ptr(cost),
                status.ctypes.data_as(_ip), iters.ctypes.data_as(_ip)))
        elif cost_params is not None:
            x_init = None if x_init is None else _f64(x_init, (B, self.num_vars))
            mult_init = None if mult_init is None else _f64(mult_init, (B, self.num_mults))
            mult = np.empty((B, self.num_mults)) if want_mult else None
            _check(self._lib.b200mpc_solve_batch_cost(
                self._h, B, _ptr(states), _ptr(coeffs), ncoef, _ptr(_cost8(cost_params, B)),
                None if x_init is None else _ptr(x_init), None if mult_init is None else _ptr(mult_init), float(mu_init),
                _ptr(out8), _ptr(traj) if want_traj else None, _ptr(mult) if want_mult else None, _ptr(cost),
                status.ctypes.data_as(_ip), iters.ctypes.data_as(_ip)))
        elif x_init is None and mult_init is None and not want_mult:
            _check(self._lib.b200mpc_solve_batch(self._h, B, _ptr(states), _ptr(coeffs), ncoef, _ptr(out8),
                                                 _ptr(traj) if want_traj else None, _ptr(cost),
                                                 status.ctypes.data_as(_ip), iters.ctypes.data_as(_ip)))
        else:
            if x_init is not None:
                x_init = _f64(x_init, (B, self.num_vars))
            if mult_init is not None:
                mult_init = _f64(mult_init, (B, self.num_mults))
            mult = np.empty((B, self.num_mults)) if want_mult else None
            _check(self._lib.b200mpc_solve_batch_warm(
                self._h, B, _ptr(states), _ptr(coeffs), ncoef, None if x_init is None else _ptr(x_init),
                None if mult_init is None else _ptr(mult_init), float(mu_init), _ptr(out8),
                _ptr(traj) if want_traj else None, _ptr(mult) if want_mult else None, _ptr(cost),
                status.ctypes.data_as(_ip), iters.ctypes.data_as(_ip)))
        r = dict(out8=out8, cost=cost, status=status, iters=iters)
        if want_traj:
            r["traj"] = traj
        if want_mult:
            r["mult"] = mult
        return r

    def solve_batch_device(self, B, d_state6, d_coeffs, ncoef, d_out8, d_traj=0, d_obj=0, d_status=0, d_iters=0,
                           stream=0):
        """Raw device-pointer call (integers), field-major buffers; asynchronous on `stream`."""
        _check(self._lib.b200mpc_solve_batch_device(self._h, B, d_state6, d_coeffs, ncoef, d_out8, d_traj or None,
                                                    d_obj or None, d_status or None, d_iters or None, stream or None))

    def solve_batch_warm_device(self, B, d_state6, d_coeffs, ncoef, d_x_init, d_mult_init, mu_init, d_out8, d_traj=0,
                                d_mult=0, d_obj=0, d_status=0, d_iters=0, stream=0):
        """Raw device-pointer warm start (integers), field-major buffers: d_x_init [8N-2][B] (0 = default start point),
        d_mult_init / d_mult [10N-4][B] (0 = none); asynchronous on `stream`.  See b200mpc_solve_batch_warm_device."""
        _check(self._lib.b200mpc_solve_batch_warm_device(self._h, B, d_state6, d_coeffs, ncoef, d_x_init or None,
                                                         d_mult_init or None, float(mu_init), d_out8, d_traj or None,
                                                         d_mult or None, d_obj or None, d_status or None, d_iters or None,
                                                         stream or None))

    def solve_batch_cost_device(self, B, d_state6, d_coeffs, ncoef, d_cost8, d_x_init=0, d_mult_init=0, mu_init=1e-4,
                                d_out8=0, d_traj=0, d_mult=0, d_obj=0, d_status=0, d_iters=0, stream=0):
        """Raw device-pointer solve with per-problem costs (integers, 0 = none), field-major buffers: d_cost8 [8][B] in
        the order PARAM_NAMES (0 = the handle's values); asynchronous on `stream`.  See b200mpc_solve_batch_cost_device."""
        _check(self._lib.b200mpc_solve_batch_cost_device(self._h, B, d_state6, d_coeffs, ncoef, d_cost8 or None,
                                                         d_x_init or None, d_mult_init or None, float(mu_init), d_out8,
                                                         d_traj or None, d_mult or None, d_obj or None, d_status or None,
                                                         d_iters or None, stream or None))

    def solve_batch_model_device(self, B, d_state6, d_coeffs, ncoef, d_cost8, d_model4, d_x_init=0, d_mult_init=0,
                                 mu_init=1e-4, d_out8=0, d_traj=0, d_mult=0, d_obj=0, d_status=0, d_iters=0, stream=0):
        """Raw device-pointer solve with per-problem costs and vehicle models (integers, 0 = none), field-major buffers:
        d_cost8 [8][B] in the order PARAM_NAMES, d_model4 [4][B] in the order MODEL_NAMES (0 = the handle's values);
        asynchronous on `stream`.  See b200mpc_solve_batch_model_device."""
        _check(self._lib.b200mpc_solve_batch_model_device(self._h, B, d_state6, d_coeffs, ncoef, d_cost8 or None,
                                                          d_model4 or None, d_x_init or None, d_mult_init or None,
                                                          float(mu_init), d_out8, d_traj or None, d_mult or None,
                                                          d_obj or None, d_status or None, d_iters or None, stream or None))

    def solve_batch_vjp(self, states, coeffs, traj, mult, g_out8=None, g_traj=None, g_obj=None, want_params=False,
                        cost_params=None, model_params=None, want_model=False):
        """Adjoint sensitivities of solutions (b200mpc_solve_batch_vjp; not reference behaviour): for a loss L with the
        incoming gradients g_out8 (B,8), g_traj (B,8N-2), g_obj (B,) -- any of them None, not all -- returns
        dict(grad_state6 (B,6), grad_coeffs (B,ncoef) per problem, status (B,), and grad_params (B,8) in the order
        PARAM_NAMES if want_params).  traj (B,8N-2) and mult (B,10N-4) must be a converged solution of (states, coeffs)
        on a handle with these params, as solve_batch(..., want_traj=True, want_mult=True) returns it.  cost_params (B,8)
        or (8,): the per-problem costs the solve used (b200mpc_solve_batch_vjp_cost); grad_params is w.r.t. them.
        model_params (B,4) or (4,): the per-problem vehicle models the solve used; want_model adds grad_model (B,4) in the
        order MODEL_NAMES, w.r.t. them or, without model_params, w.r.t. the handle's (b200mpc_solve_batch_vjp_model)."""
        states = _f64(states)
        if states.ndim != 2 or states.shape[1] != 6:
            raise ValueError("states must be (B, 6)")
        B = states.shape[0]
        coeffs = _f64(coeffs)
        if coeffs.ndim == 1:
            coeffs = np.ascontiguousarray(np.broadcast_to(coeffs, (B, coeffs.size)))
        if coeffs.shape[0] != B:
            raise ValueError("coeffs must be (B, ncoef)")
        ncoef = coeffs.shape[1]
        traj = _f64(traj, (B, self.num_vars))
        mult = _f64(mult, (B, self.num_mults))
        g_out8 = None if g_out8 is None else _f64(g_out8, (B, 8))
        g_traj = None if g_traj is None else _f64(g_traj, (B, self.num_vars))
        g_obj = None if g_obj is None else _f64(g_obj, (B,))
        gs = np.empty((B, 6)); gc = np.empty((B, ncoef)); gp = np.empty((B, 8)) if want_params else None
        status = np.empty(B, dtype=np.int32)
        grads = (None if g_out8 is None else _ptr(g_out8), None if g_traj is None else _ptr(g_traj),
                 None if g_obj is None else _ptr(g_obj), _ptr(gs), _ptr(gc), None if gp is None else _ptr(gp),
                 status.ctypes.data_as(_ip))
        gm = np.empty((B, 4)) if want_model else None
        if model_params is not None or want_model:
            c8 = None if cost_params is None else _cost8(cost_params, B)
            m4 = None if model_params is None else _model4(model_params, B)
            _check(self._lib.b200mpc_solve_batch_vjp_model(
                self._h, B, _ptr(states), _ptr(coeffs), ncoef, None if c8 is None else _ptr(c8),
                None if m4 is None else _ptr(m4), _ptr(traj), _ptr(mult), *grads[:6], None if gm is None else _ptr(gm),
                grads[6]))
        elif cost_params is None:
            _check(self._lib.b200mpc_solve_batch_vjp(self._h, B, _ptr(states), _ptr(coeffs), ncoef, _ptr(traj), _ptr(mult),
                                                     *grads))
        else:
            _check(self._lib.b200mpc_solve_batch_vjp_cost(self._h, B, _ptr(states), _ptr(coeffs), ncoef,
                                                          _ptr(_cost8(cost_params, B)), _ptr(traj), _ptr(mult), *grads))
        r = dict(grad_state6=gs, grad_coeffs=gc, status=status)
        if want_params:
            r["grad_params"] = gp
        if want_model:
            r["grad_model"] = gm
        return r

    def solve_batch_vjp_device(self, B, d_state6, d_coeffs, ncoef, d_traj, d_mult, d_g_out8=0, d_g_traj=0, d_g_obj=0,
                               d_grad_state6=0, d_grad_coeffs=0, d_grad_params=0, d_status=0, stream=0):
        """Raw device-pointer VJP (integers, 0 = none), field-major buffers; one kernel launch, asynchronous on `stream`.
        See b200mpc_solve_batch_vjp_device."""
        _check(self._lib.b200mpc_solve_batch_vjp_device(self._h, B, d_state6, d_coeffs, ncoef, d_traj, d_mult,
                                                        d_g_out8 or None, d_g_traj or None, d_g_obj or None,
                                                        d_grad_state6 or None, d_grad_coeffs or None, d_grad_params or None,
                                                        d_status or None, stream or None))

    def solve_batch_vjp_cost_device(self, B, d_state6, d_coeffs, ncoef, d_cost8, d_traj, d_mult, d_g_out8=0, d_g_traj=0,
                                    d_g_obj=0, d_grad_state6=0, d_grad_coeffs=0, d_grad_params=0, d_status=0, stream=0):
        """Raw device-pointer VJP with per-problem costs (integers, 0 = none), field-major buffers, d_cost8 [8][B]; one
        kernel launch, asynchronous on `stream`.  See b200mpc_solve_batch_vjp_cost_device."""
        _check(self._lib.b200mpc_solve_batch_vjp_cost_device(self._h, B, d_state6, d_coeffs, ncoef, d_cost8 or None, d_traj,
                                                             d_mult, d_g_out8 or None, d_g_traj or None, d_g_obj or None,
                                                             d_grad_state6 or None, d_grad_coeffs or None,
                                                             d_grad_params or None, d_status or None, stream or None))

    def solve_batch_vjp_model_device(self, B, d_state6, d_coeffs, ncoef, d_cost8, d_model4, d_traj, d_mult, d_g_out8=0,
                                     d_g_traj=0, d_g_obj=0, d_grad_state6=0, d_grad_coeffs=0, d_grad_params=0, d_grad_model=0,
                                     d_status=0, stream=0):
        """Raw device-pointer VJP with per-problem costs and vehicle models (integers, 0 = none), field-major buffers,
        d_cost8 [8][B], d_model4 / d_grad_model [4][B]; one kernel launch, asynchronous on `stream`.  See
        b200mpc_solve_batch_vjp_model_device."""
        _check(self._lib.b200mpc_solve_batch_vjp_model_device(self._h, B, d_state6, d_coeffs, ncoef, d_cost8 or None,
                                                              d_model4 or None, d_traj, d_mult, d_g_out8 or None,
                                                              d_g_traj or None, d_g_obj or None, d_grad_state6 or None,
                                                              d_grad_coeffs or None, d_grad_params or None,
                                                              d_grad_model or None, d_status or None, stream or None))

    def solve_batch_jvp(self, states, coeffs, traj, mult, t_state6=None, t_coeffs=None, t_cost=None, t_model=None,
                        cost_params=None, model_params=None):
        """Forward sensitivities of solutions (b200mpc_solve_batch_jvp; not reference behaviour): the derivative of each
        problem's (out8, traj, obj) along the tangent t_state6 (B,6), t_coeffs (B,ncoef) or (ncoef,), t_cost (B,8) or (8,)
        in the order PARAM_NAMES, t_model (B,4) or (4,) in the order MODEL_NAMES -- any of them None (zero), not all.
        Returns dict(t_out8 (B,8), t_traj (B,8N-2), t_obj (B,), status (B,)).  states, coeffs, traj, mult, cost_params
        and model_params as for solve_batch_vjp; t_cost / t_model are w.r.t. the per-problem rows or, without them, the
        handle's values."""
        states = _f64(states)
        if states.ndim != 2 or states.shape[1] != 6:
            raise ValueError("states must be (B, 6)")
        B = states.shape[0]
        coeffs = _f64(coeffs)
        if coeffs.ndim == 1:
            coeffs = np.ascontiguousarray(np.broadcast_to(coeffs, (B, coeffs.size)))
        if coeffs.ndim != 2 or coeffs.shape[0] != B:
            raise ValueError("coeffs must be (B, ncoef) or (ncoef,)")
        ncoef = coeffs.shape[1]
        traj = _f64(traj, (B, self.num_vars))
        mult = _f64(mult, (B, self.num_mults))
        if t_state6 is not None:
            t_state6 = _f64(t_state6)
            if t_state6.shape != (B, 6):
                raise ValueError("t_state6 must be (B, 6)")
        if t_coeffs is not None:
            t_coeffs = _f64(t_coeffs)
            if t_coeffs.ndim == 1:
                t_coeffs = np.broadcast_to(t_coeffs, (B, t_coeffs.size))
            if t_coeffs.shape != (B, ncoef):
                raise ValueError("t_coeffs must be (B, ncoef) or (ncoef,), ncoef as coeffs")
            t_coeffs = np.ascontiguousarray(t_coeffs)
        t_cost = None if t_cost is None else _cost8(t_cost, B)
        t_model = None if t_model is None else _model4(t_model, B)
        c8 = None if cost_params is None else _cost8(cost_params, B)
        m4 = None if model_params is None else _model4(model_params, B)
        t_out8, t_traj, t_obj = np.empty((B, 8)), np.empty((B, self.num_vars)), np.empty(B)
        status = np.empty(B, dtype=np.int32)
        opt = lambda a: None if a is None else _ptr(a)
        _check(self._lib.b200mpc_solve_batch_jvp(
            self._h, B, _ptr(states), _ptr(coeffs), ncoef, opt(c8), opt(m4), _ptr(traj), _ptr(mult), opt(t_state6),
            opt(t_coeffs), opt(t_cost), opt(t_model), _ptr(t_out8), _ptr(t_traj), _ptr(t_obj), status.ctypes.data_as(_ip)))
        return dict(t_out8=t_out8, t_traj=t_traj, t_obj=t_obj, status=status)

    def solve_batch_jvp_device(self, B, d_state6, d_coeffs, ncoef, d_cost8, d_model4, d_traj, d_mult, d_t_state6=0,
                               d_t_coeffs=0, d_t_cost8=0, d_t_model4=0, d_t_out8=0, d_t_traj=0, d_t_obj=0, d_status=0,
                               stream=0):
        """Raw device-pointer JVP (integers, 0 = none), field-major buffers, d_cost8 [8][B], d_model4 / d_t_model4 [4][B];
        one kernel launch, asynchronous on `stream`.  See b200mpc_solve_batch_jvp_device."""
        _check(self._lib.b200mpc_solve_batch_jvp_device(self._h, B, d_state6, d_coeffs, ncoef, d_cost8 or None,
                                                        d_model4 or None, d_traj, d_mult, d_t_state6 or None,
                                                        d_t_coeffs or None, d_t_cost8 or None, d_t_model4 or None,
                                                        d_t_out8 or None, d_t_traj or None, d_t_obj or None,
                                                        d_status or None, stream or None))

    def wait(self):
        """Waits for everything queued on this handle's own stream (b200mpc_solve_batch_async calls)."""
        _check(self._lib.b200mpc_wait(self._h))

    def closed_loop(self, states, coeffs, steps):
        """solution/main.cpp:51-76 for B vehicles: returns dict(hist8 (steps,B,8), cost (steps,B), iters (steps,B))."""
        states = _f64(states)
        if states.ndim == 1:
            states = states[None, :]
        B = states.shape[0]
        coeffs = _f64(coeffs)
        if coeffs.ndim == 1:
            coeffs = np.ascontiguousarray(np.broadcast_to(coeffs, (B, coeffs.size)))
        hist = np.empty((steps, B, 8))
        cost = np.empty((steps, B))
        iters = np.empty((steps, B), dtype=np.int32)
        _check(self._lib.b200mpc_closed_loop_batch(self._h, B, steps, _ptr(states), _ptr(coeffs), coeffs.shape[1],
                                                   _ptr(hist), _ptr(cost), iters.ctypes.data_as(_ip)))
        return dict(hist8=hist, cost=cost, iters=iters)

    def set_solver_mode(self, mode=0, rounds=0, fused_below=-1):
        """mode 0 = per-pass kernels (default), 1 = fused kernel; see include/b200mpc.h."""
        _check(self._lib.b200mpc_set_solver_mode(self._h, mode, rounds, fused_below))

    def set_batch_split(self, parts):
        """Cut large batches into `parts` (1..4) sub-batches that run concurrently inside one call (default 4; use 1
        when the caller overlaps several calls itself)."""
        _check(self._lib.b200mpc_set_batch_split(self._h, int(parts)))

    def set_restoration(self, mode=2):
        """What follows a failed line search: 0 = status -2 at the iteration where the reference's Ipopt enters its
        restoration phase, 1 = the restoration step, 2 (the library default) = Ipopt's soft restoration phase first,
        then the restoration step.  See b200mpc_set_restoration."""
        _check(self._lib.b200mpc_set_restoration(self._h, int(mode)))

    def set_compaction(self, max_live_fraction=0.7, from_round=4):
        """Throughput path: after every round from `from_round` on, move the unfinished problems to consecutive
        workspace slots when they fill at most this fraction of the occupied slots (0 = off)."""
        _check(self._lib.b200mpc_set_compaction(self._h, float(max_live_fraction), int(from_round)))

    def set_handover(self, occupied_slots=1184, from_round=14):
        """Occupied workspace slots at which the cooperative kernel takes the rest of a batch over (default 1184: best for
        one call at a time; 64-256 for a caller that overlaps several calls).  See b200mpc_set_handover."""
        _check(self._lib.b200mpc_set_handover(self._h, int(occupied_slots), int(from_round)))

    def set_pipeline(self, depth=8, tail_slots=4096):
        """Pipelined solves: solve_batch_device calls issued on different streams overlap on this one handle -- the
        bulk of a batch runs in the full-size workspace, its last `tail_slots` unfinished problems finish in one of
        `depth` small tail contexts while the next batch's bulk runs (0 = off).  See b200mpc_set_pipeline."""
        _check(self._lib.b200mpc_set_pipeline(self._h, int(depth), int(tail_slots)))

    def set_warm_start(self, enable=True, mu_init=1e-4):
        """closed_loop() only (solve_batch takes x_init / mult_init instead): steps after the first start from the shifted previous solution (not reference behaviour)."""
        _check(self._lib.b200mpc_set_warm_start(self._h, int(enable), float(mu_init)))

    # -- measurement helpers
    def set_timing(self, enable=True):
        """Bracket every solve with CUDA events (read them with kernel_time_ms); off by default."""
        _check(self._lib.b200mpc_set_timing(self._h, int(enable)))

    def kernel_time_ms(self, reset=True):
        t = ctypes.c_double()
        n = ctypes.c_int()
        _check(self._lib.b200mpc_kernel_time_ms(self._h, ctypes.byref(t), ctypes.byref(n), int(reset)))
        return t.value, n.value

    def fp64_peak_tflops(self):
        t = ctypes.c_double()
        _check(self._lib.b200mpc_measure_fp64_peak(self._h, ctypes.byref(t)))
        return t.value

    def selftest_division(self, a, b):
        """(a / b, 1 / b) as the solver's sweeps compute them on the device (b200mpc_selftest_division)."""
        a = np.ascontiguousarray(a, dtype=np.float64)
        b = np.ascontiguousarray(b, dtype=np.float64)
        assert a.shape == b.shape and a.ndim == 1
        q, r = np.empty_like(a), np.empty_like(a)
        _check(self._lib.b200mpc_selftest_division(self._h, len(a), a.ctypes.data_as(_dp), b.ctypes.data_as(_dp),
                                                   q.ctypes.data_as(_dp), r.ctypes.data_as(_dp)))
        return q, r

    def launch_count(self):
        return int(self._lib.b200mpc_launch_count(self._h))


def _shift_index(N, mult):
    """Source index of every entry of a solution (mult=False: 8N-2 variables, True: 10N-4 multipliers) shifted by one
    stage: entry t of each per-stage block takes entry t+1, the last stage is repeated."""
    M = N - 1
    st = np.minimum(np.arange(N) + 1, N - 1)
    ct = np.minimum(np.arange(M) + 1, M - 1)
    blocks = [k * N + st for k in range(6)] + [6 * N + j * M + ct for j in range(4 if mult else 2)]
    return np.concatenate(blocks)


def shift_solution(traj, mult, N, field_major=None):
    """One receding-horizon step: the solution (traj (8N-2 per problem), mult (10N-4 per problem) or None) shifted by one
    stage -- states, controls and multipliers of stage t+1 move to stage t, the last stage is repeated -- as x_init /
    mult_init of the next step's warm-started solve.  NumPy arrays or torch tensors (on any device: the shift runs
    there), per-problem rows (B, 8N-2) as solve_batch returns them or field-major (8N-2, B) as the device entry points
    use; field_major=None infers the layout from the shape.  Returns (x_init, mult_init) of the same kind and layout."""
    nv = 8 * N - 2

    def layout(a, n):
        if field_major is not None:
            return bool(field_major)
        rows = a.ndim >= 1 and a.shape[-1] == n
        fields = a.ndim == 2 and a.shape[0] == n
        if rows == fields:
            raise ValueError(f"cannot tell the layout of an array of shape {tuple(a.shape)}: pass field_major")
        return fields

    def shift(a, n, is_mult):
        if a is None:
            return None
        if a.shape[0 if layout(a, n) else -1] != n:
            raise ValueError(f"expected {n} entries per problem, got shape {tuple(a.shape)}")
        idx = _shift_index(N, is_mult)
        dim = 0 if layout(a, n) else a.ndim - 1
        if isinstance(a, np.ndarray):
            return np.ascontiguousarray(np.take(a, idx, axis=dim))
        import torch
        return a.index_select(dim, torch.as_tensor(idx, device=a.device)).contiguous()

    return shift(traj, nv, False), shift(mult, 10 * N - 4, True)


def solve_batch_multi(mpcs, states, coeffs, want_traj=False):
    """One batch sharded by contiguous index ranges over several MPC handles (one per device)."""
    lib = load_library()
    states = _f64(states)
    B = states.shape[0]
    coeffs = _f64(coeffs)
    if coeffs.ndim == 1:
        coeffs = np.ascontiguousarray(np.broadcast_to(coeffs, (B, coeffs.size)))
    hs = (_vp * len(mpcs))(*[m.handle for m in mpcs])
    out8 = np.empty((B, 8)); cost = np.empty(B)
    status = np.empty(B, dtype=np.int32); iters = np.empty(B, dtype=np.int32)
    traj = np.empty((B, mpcs[0].num_vars)) if want_traj else None
    _check(lib.b200mpc_solve_batch_multi(hs, len(mpcs), B, _ptr(states), _ptr(coeffs), coeffs.shape[1], _ptr(out8),
                                         _ptr(traj) if want_traj else None, _ptr(cost), status.ctypes.data_as(_ip),
                                         iters.ctypes.data_as(_ip)))
    r = dict(out8=out8, cost=cost, status=status, iters=iters)
    if want_traj:
        r["traj"] = traj
    return r


# ---------------------------------------------------------------------------------------------
# helpers.h / globalKinematic.  They need a device handle; a process-wide default one is created lazily.
_default = None


def _default_mpc():
    global _default
    if _default is None:
        _default = MPC()
    return _default


def polyfit_batch(xs, ys, order, mpc=None):
    """B fits at once: xs, ys (B, m) -> coeffs (B, order+1), ascending powers."""
    m_ = mpc or _default_mpc()
    xs = _f64(xs); ys = _f64(ys)
    if xs.shape != ys.shape or xs.ndim != 2:
        raise ValueError("xs and ys must both be (B, m)")
    B, m = xs.shape
    out = np.empty((B, order + 1))
    _check(m_._lib.b200mpc_polyfit_batch(m_.handle, B, _ptr(xs), _ptr(ys), m, order, _ptr(out)))
    return out


def polyfit(xvals, yvals, order, mpc=None):
    """helpers.h:24-44.  Like the reference's assert (helpers.h:25-26) sizes must match and 1 <= order <= m-1."""
    xvals = _f64(xvals).ravel(); yvals = _f64(yvals).ravel()
    assert xvals.size == yvals.size
    assert 1 <= order <= xvals.size - 1
    return polyfit_batch(xvals[None, :], yvals[None, :], order, mpc)[0]


def polyeval_batch(coeffs, x, mpc=None):
    m_ = mpc or _default_mpc()
    coeffs = _f64(coeffs); x = _f64(x).ravel()
    B = x.size
    if coeffs.ndim == 1:
        coeffs = np.ascontiguousarray(np.broadcast_to(coeffs, (B, coeffs.size)))
    y = np.empty(B)
    _check(m_._lib.b200mpc_polyeval_batch(m_.handle, B, _ptr(coeffs), coeffs.shape[1], _ptr(x), _ptr(y)))
    return y


def polyeval(coeffs, x, mpc=None):
    """helpers.h:13-19."""
    return float(polyeval_batch(_f64(coeffs).ravel(), [x], mpc)[0])


def rollout_batch(states, actuators, dt, Lf=2.0, mpc=None):
    """states (B,4), actuators (B,H,2) -> (B,H,4): the state after each of H Euler steps."""
    m_ = mpc or _default_mpc()
    states = _f64(states); actuators = _f64(actuators)
    if actuators.ndim == 2:
        actuators = actuators[:, None, :]
    B, H = actuators.shape[0], actuators.shape[1]
    if states.shape != (B, 4) or actuators.shape[2] != 2:
        raise ValueError("states must be (B,4) and actuators (B,H,2)")
    actuators = np.ascontiguousarray(actuators)
    out = np.empty((B, H, 4))
    _check(m_._lib.b200mpc_rollout_batch(m_.handle, B, H, _ptr(states), _ptr(actuators), float(dt), float(Lf), _ptr(out)))
    return out


def roadmap_reference_batch(poses, centerline, mpc=None):
    """Roadmap front-end: poses (B,4) = (x, y, psi, v) in the road's global frame, centerline (n_wp,2) ->
    (state6 (B,6), coeffs (B,4)) in the vehicle frame, ready for MPC.solve_batch."""
    m_ = mpc or _default_mpc()
    poses = _f64(poses); centerline = _f64(centerline)
    if poses.ndim != 2 or poses.shape[1] != 4 or centerline.ndim != 2 or centerline.shape[1] != 2:
        raise ValueError("poses must be (B,4) and centerline (n_wp,2)")
    B = poses.shape[0]
    st = np.empty((B, 6)); cf = np.empty((B, 4))
    _check(m_._lib.b200mpc_roadmap_reference_batch(m_.handle, B, _ptr(poses), _ptr(centerline), centerline.shape[0], _ptr(st), _ptr(cf)))
    return st, cf


def read_roadmap_csv(path, float_fields=False):
    """The reference's roadmap file (7 numbers per line) -> (centerline (n_wp, 2), slope (n_wp,)), parsed by the library's
    host-side reader (b200mpc_read_roadmap_csv).  float_fields=True converts every field through single precision like
    the reference's std::stof (mpc_to_line/src/custom_MPC.h:35-44)."""
    lib = load_library()
    n = ctypes.c_int()
    _check(lib.b200mpc_read_roadmap_csv(os.fsencode(path), int(float_fields), None, None, 0, ctypes.byref(n)))
    cl = np.empty((n.value, 2)); sl = np.empty(n.value)
    _check(lib.b200mpc_read_roadmap_csv(os.fsencode(path), int(float_fields), _ptr(cl), _ptr(sl), n.value, ctypes.byref(n)))
    return cl, sl


def global_kinematic(state, actuators, dt, Lf=2.0, mpc=None):
    """global_kinematic_model/solution/main.cpp:36-62 (Lf = 2 there, :15)."""
    return rollout_batch(_f64(state).reshape(1, 4), _f64(actuators).reshape(1, 1, 2), dt, Lf, mpc)[0, 0]
