"""-m "not gpu": the init kernel's cold start (Solver::kernel_ls_round) runs the multiplier-initialisation round on the
start point in closed form instead of leaving it to a round of the per-pass sweeps, which read the start point back from
the workspace.  The host build of the solver core (tests/hostsim/hostsim_cold.cpp) runs both on the same problem: the
workspace after the round (scalar record, iterate, Riccati factors, direction) and the final solution must be the same
bits, for the discarded estimate (ref_v = 40) and for the kept one (F_LSKEEP, small ref_v), across horizons and with
non-default cost and vehicle-model parameters."""
import ctypes
import os

import numpy as np
import pytest

import oracle_bindings as ob
from conftest import ROOT, golden

# the horizons test_horizons.py holds the host build to
CPU_N = [2, 3, 4, 5, 6, 7, 9, 16, 31, 32, 33, 51, 52, 64, 65, 68, 69, 102, 103, 204, 205]


@pytest.fixture(scope="module")
def cold(_build_everything):
    dp, ip = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int)
    lib = ctypes.CDLL(os.path.join(ROOT, "tests", "hostsim", "libhostsim_cold.so"))

    def run(state6, coeffs, **params):
        p = ob.default_params(**params)
        N = p.N
        n = 83 * (N + 2)   # workspace_doubles_per_problem
        st = np.ascontiguousarray(state6, dtype=np.float64)
        cf = np.ascontiguousarray(coeffs, dtype=np.float64)
        ws = np.zeros((2, n)); o8 = np.zeros((2, 8)); obj = np.zeros(2); x = np.zeros((2, 8 * N - 2))
        it = np.zeros(2, dtype=np.int32); status = np.zeros(2, dtype=np.int32); kept = ctypes.c_int()
        rc = lib.hostsim_cold_compare(ctypes.byref(p), st.ctypes.data_as(dp), cf.ctypes.data_as(dp), len(cf),
                                      ws.ctypes.data_as(dp), o8.ctypes.data_as(dp), obj.ctypes.data_as(dp),
                                      it.ctypes.data_as(ip), status.ctypes.data_as(ip), x.ctypes.data_as(dp), ctypes.byref(kept))
        assert rc == 0
        # bits, not values: the rows neither path writes are NaN in both
        np.testing.assert_array_equal(ws[0].view(np.uint64), ws[1].view(np.uint64))
        np.testing.assert_array_equal(o8[0].view(np.uint64), o8[1].view(np.uint64))
        np.testing.assert_array_equal(x[0].view(np.uint64), x[1].view(np.uint64))
        assert obj[0].tobytes() == obj[1].tobytes() and it[0] == it[1] and status[0] == status[1]
        return dict(kept=bool(kept.value), status=int(status[0]), iters=int(it[0]))
    return run


@pytest.mark.parametrize("name", ["line_256.npz", "roadmap_256.npz"])
def test_goldens(cold, name):
    g = golden(name)
    cf = g["coeffs"] if "coeffs" in g.files else g["fit"]
    for b in range(256):
        r = cold(g["states"][b], cf[b])
        assert not r["kept"]   # ref_v = 40: the estimate exceeds constr_mult_init_max
        assert r["status"] == g["status"][b]


@pytest.mark.parametrize("N", CPU_N)
def test_horizons(cold, N):
    g, gl = golden("roadmap_256.npz"), golden("line_256.npz")
    probs = [(g["states"][b], g["fit"][b]) for b in (0, 64)] + [(gl["states"][b], gl["coeffs"][b]) for b in (0, 96)]
    if N > 103:
        probs = probs[:1] if N % 2 == 0 else probs[2:3]
    for st, cf in probs:
        cold(st, cf, N=N)


def test_cost_and_model_parameters(cold):
    """Cost weights and ref_v change df and the LS right-hand side; dt, Lf and the actuator bounds change the dynamics
    and u_init, the controls of the start point."""
    g = golden("line_256.npz")
    sets = [dict(w_cte=3.0, w_epsi=0.5, w_v=0.2, w_delta=10.0, w_a=2.0, w_ddelta=50.0, w_da=4.0),
            dict(ref_v=25.0, w_v=4.0),
            dict(dt=0.08, Lf=3.1, delta_max=0.3, a_max=2.5),
            dict(dt=0.04, Lf=2.2, delta_max=0.6, a_max=0.5, w_cte=2.0, ref_v=30.0),
            dict(delta_max=0.2, a_max=4.0, N=50)]
    for kw in sets:
        for b in range(0, 256, 32):
            cold(g["states"][b], g["coeffs"][b], **kw)


def test_kept_estimate(cold):
    """ref_v = 6 with speeds near it: the estimate stays below 1000 and is stored by a second step pass."""
    g = golden("line_256.npz")
    n_kept = 0
    for b in range(32):
        st = g["states"][b].copy()
        st[3] = 5.0 + 0.2 * (b % 6)
        for N in (25, 7, 60):
            n_kept += cold(st, g["coeffs"][b], ref_v=6.0, N=N)["kept"]
    assert n_kept >= 48, n_kept
