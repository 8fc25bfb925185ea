"""Forward sensitivities of solutions (b200mpc_solve_batch_jvp, not reference behaviour).  CPU tests run the host build
of the solver core (tests/hostsim/hostsim_jvp.cpp) against the VJP's host build (the adjoint identity <v, J u> =
<J^T v, u>), a dense KKT solve built from the C port's evaluator and finite differences of the host-build solve; -m gpu
runs the library's kernel against the host build and the device VJP and checks the C ABI, the Python API and forward-mode
AD through the autograd wrapper."""
import ctypes
import os
import sys
import types

import numpy as np
import pytest

from conftest import ROOT, golden, has_gpu
from test_cost_params import _kw, _random_costs, _weight_sets
from test_model_params import LINE_N, LINE_REF_V, MNAMES, MODEL_ROWS, _line_problems, _mkw, _random_models
from test_sensitivity import PNAMES, _coeffs, _problems

dp = ctypes.POINTER(ctypes.c_double)
CF_SCALE = np.array([1e-1, 1e-2, 1e-4, 1e-6])   # tangent scale of the coefficients (|x| up to ~100)


def _p(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float64).ctypes.data_as(dp)


@pytest.fixture(scope="module")
def host(_build_everything):
    """solve(state6, coeffs, **params): the host build's solve with its multipliers (hostsim_solve_guess from the
    default start); vjp(...): hostsim_vjp_model; jvp(...): hostsim_jvp, one problem each."""
    import oracle_bindings as ob
    hs = os.path.join(ob.ROOT, "tests", "hostsim")
    lg = ctypes.CDLL(os.path.join(hs, "libhostsim_guess.so"))
    lm = ctypes.CDLL(os.path.join(hs, "libhostsim_sens_model.so"))
    lm.hostsim_vjp_model.argtypes = [ctypes.c_void_p, dp, dp, ctypes.c_int, dp, dp, dp, dp, ctypes.c_double, dp, dp, dp, dp]
    lj = ctypes.CDLL(os.path.join(hs, "libhostsim_jvp.so"))
    lj.hostsim_jvp.argtypes = [ctypes.c_void_p, dp, dp, ctypes.c_int, dp, dp, dp, dp, dp, dp, dp, dp, dp]

    class H:
        @staticmethod
        def solve(state6, coeffs, **params):
            p = ob.default_params(**params)
            N = p.N
            st = np.ascontiguousarray(state6, dtype=np.float64); c = np.ascontiguousarray(coeffs, dtype=np.float64)
            x = np.zeros(8 * N - 2); o8 = np.zeros(8); obj = ctypes.c_double(); it = ctypes.c_int(); m = np.zeros(10 * N - 4)
            rc = lg.hostsim_solve_guess(ctypes.byref(p), _p(st), _p(c), len(c), None, None, ctypes.c_double(1e-4), _p(x),
                                        _p(o8), ctypes.byref(obj), ctypes.byref(it), _p(m), 0)
            return dict(status=rc, x=x, out8=o8, obj=obj.value, iters=it.value, mult=m)

        @staticmethod
        def vjp(state6, coeffs, x, mult, g_out8=None, g_traj=None, g_obj=0.0, **params):
            p = ob.default_params(**params)
            gs, gc, gp, gm = np.zeros(6), np.zeros(len(coeffs)), np.zeros(8), np.zeros(4)
            rc = lm.hostsim_vjp_model(ctypes.byref(p), _p(state6), _p(coeffs), len(coeffs), _p(x), _p(mult), _p(g_out8),
                                      _p(g_traj), float(g_obj), _p(gs), _p(gc), _p(gp), _p(gm))
            return dict(status=rc, grad_state6=gs, grad_coeffs=gc, grad_params=gp, grad_model=gm)

        @staticmethod
        def jvp(state6, coeffs, x, mult, t_state6=None, t_coeffs=None, t_cost=None, t_model=None, **params):
            p = ob.default_params(**params)
            a = [None if v is None else np.ascontiguousarray(v, dtype=np.float64)
                 for v in (state6, coeffs, x, mult, t_state6, t_coeffs, t_cost, t_model)]
            to8, tt, tob = np.zeros(8), np.zeros(8 * p.N - 2), ctypes.c_double()
            rc = lj.hostsim_jvp(ctypes.byref(p), _p(a[0]), _p(a[1]), len(a[1]), *[_p(v) for v in a[2:]], _p(to8), _p(tt),
                                ctypes.byref(tob))
            return dict(status=rc, t_out8=to8, t_traj=tt, t_obj=tob.value)
    return H


def _tangent(rng, ncoef, p8, m4):
    """A random tangent of all four groups, scaled to the inputs: state6, coefficients (CF_SCALE), cost8 and model4
    relative to their values."""
    return (rng.standard_normal(6), rng.standard_normal(ncoef) * CF_SCALE[:ncoef], rng.standard_normal(8) * p8,
            rng.standard_normal(4) * m4)


def _identity(host, st, cf, r, rng, p8, m4, **kw):
    """|<v, J u> - <J^T v, u>| and the sum of the magnitudes of the terms, for random u and v."""
    N = kw.get("N", 25)
    u = _tangent(rng, len(cf), p8, m4)
    go8, gt, gob = rng.standard_normal(8), rng.standard_normal(8 * N - 2), float(rng.standard_normal())
    j = host.jvp(st, cf, r["x"], r["mult"], *u, **kw)
    v = host.vjp(st, cf, r["x"], r["mult"], go8, gt, gob, **kw)
    assert j["status"] == 0 and v["status"] == 0
    lhs = np.concatenate([go8 * j["t_out8"], gt * j["t_traj"], [gob * j["t_obj"]]])
    rhs = np.concatenate([v[k] * t for k, t in zip(("grad_state6", "grad_coeffs", "grad_params", "grad_model"), u)])
    return abs(lhs.sum() - rhs.sum()), np.abs(lhs).sum() + np.abs(rhs).sum()


def _cases():
    """(state6, coeffs, params): the 32 problems of test_sensitivity at the defaults, 4 weights_64 problems at each of
    its four cost rows, 4 line_params_64 problems at each of four model rows."""
    out = [(st, cf, {}) for st, cf in _problems()]
    g = golden("weights_64.npz")
    for c8 in _weight_sets():
        for kind, b in (("line", 0), ("line", 9), ("road", 3), ("road", 20)):
            out.append((g[f"{kind}_states"][b], g[f"{kind}_coeffs"][b], _kw(c8)))
    for m4 in MODEL_ROWS[:3]:
        for st, cf in _line_problems():
            out.append((st, cf, dict(N=LINE_N, ref_v=LINE_REF_V, **_mkw(m4))))
    return out


def _p8m4(kw):
    import oracle_bindings as ob
    p = ob.default_params(**kw)
    return np.array([getattr(p, n) for n in PNAMES]), np.array([getattr(p, n) for n in MNAMES])


# ------------------------------------------------------------------------------------------------ CPU (host build)
def test_adjoint_identity_of_the_host_build(host):
    """<v, JVP(u)> = <VJP(v), u> for random tangents on all four groups and random cotangents on out8, traj and obj."""
    rng = np.random.default_rng(31)
    worst = 0.0
    for st, cf, kw in _cases():
        r = host.solve(st, cf, **kw)
        assert r["status"] == 0, kw
        p8, m4 = _p8m4(kw)
        d, s = _identity(host, st, cf, r, rng, p8, m4, **kw)
        worst = max(worst, d / s)
    print(f"adjoint identity, host build: max |<v, Ju> - <J^T v, u>| / sum |terms| = {worst:.2e}")
    assert worst <= 1e-10, worst


@pytest.mark.parametrize("N", [2, 3, 33, 205])
def test_adjoint_identity_at_every_horizon(host, N):
    rng = np.random.default_rng(N)
    g = golden("roadmap_256.npz")
    worst, n = 0.0, 0
    for b in (0, 17, 99):
        st, cf = g["states"][b], g["fit"][b]
        r = host.solve(st, cf, N=N)
        if r["status"] != 0:
            continue
        p8, m4 = _p8m4(dict(N=N))
        d, s = _identity(host, st, cf, r, rng, p8, m4, N=N)
        worst = max(worst, d / s)
        n += 1
    assert n >= 2
    print(f"adjoint identity at N = {N}: {worst:.2e}")
    assert worst <= 1e-10, worst


def dense_jvp(state6, coeffs, x, mult, u, N=25, h=1e-6, **params):
    """dx = -K~^-1 dF~/dtheta dtheta with the full KKT system in (x, lambda, z_L, z_U) of test_model_params'
    dense_model_vjp, assembled from the C port's evaluator.  dF/dtheta dtheta of the stationarity and constraint rows is a
    directional central difference of the residual map (Richardson-extrapolated); state6 enters the rows of t = 0 (-I),
    the bounds the complementarity rows.  t_obj: df/dtheta + lambda^T dc/dtheta + dLagrangian/dbounds."""
    import oracle_bindings as ob
    ts6, tcf, tc8, tm4 = u
    p = ob.default_params(N=N, **params)
    M, n, m, nu = N - 1, 8 * N - 2, 6 * N, 2 * (N - 1)
    lam, zl, zu = mult[:m], mult[m:m + nu], mult[m + nu:]
    th0 = {k: getattr(p, k) for k in PNAMES + MNAMES[:2]}
    tth = dict(zip(PNAMES + MNAMES[:2], list(tc8) + list(tm4[:2])))

    def ev(a):
        kw = {k: th0[k] + a * tth[k] for k in th0}
        f, grad, g, J, H = ob.port_eval(x, lam, np.asarray(coeffs) + a * np.asarray(tcf),
                                        params=ob.default_params(N=N, **{**params, **kw}))
        return f, np.concatenate([grad + J.T @ lam, g]), g, J, H

    def cd(hh):
        (fp, Fp, gp, _, _), (fm, Fm, gm, _, _) = ev(hh), ev(-hh)
        return (Fp - Fm) / (2 * hh), (fp - fm) / (2 * hh) + lam @ (gp - gm) / (2 * hh)
    (dF1, e1), (dF2, e2) = cd(h), cd(h / 2)
    dF, env = (4.0 * dF2 - dF1) / 3.0, (4.0 * e2 - e1) / 3.0
    _, _, _, J, H = ev(0.0)
    W = np.tril(H) + np.tril(H, -1).T
    b = np.repeat([p.delta_max, p.a_max], M)
    rel = 1e-8 * np.maximum(1.0, b)
    xl, xu = -b - rel, b + rel
    uu = x[6 * N:]
    iu, izl, izu = 6 * N + np.arange(nu), n + m + np.arange(nu), n + m + nu + np.arange(nu)
    K = np.zeros((n + m + 2 * nu, n + m + 2 * nu))
    K[:n, :n] = W
    K[:n, n:n + m] = J.T
    K[n:n + m, :n] = J
    K[iu, izl] = -1.0
    K[iu, izu] = 1.0
    K[izl, iu] = zl
    K[izl, izl] = uu - xl
    K[izu, iu] = -zu
    K[izu, izu] = xu - uu
    rhs = np.zeros(n + m + 2 * nu)
    rhs[:n + m] = -dF
    rows0 = np.arange(6) * N
    rhs[n + rows0] += ts6            # d(s_0 - state6) = -d state6
    env -= lam[rows0] @ ts6
    db = np.repeat([(1.0 + (1e-8 if abs(bj) > 1.0 else 0.0)) * t for bj, t in zip((p.delta_max, p.a_max), tm4[2:])], M)
    rhs[izl] -= zl * db              # d(z_L (u - x_L)) = -z_L dx_L = z_L db
    rhs[izu] -= zu * db              # d(z_U (x_U - u)) = z_U dx_U
    env -= ((zl + zu) * db).sum()
    dx = np.linalg.solve(K, rhs)[:n]
    return dict(t_traj=dx, t_out8=np.concatenate([dx[np.arange(6) * N + 1], [dx[6 * N], dx[6 * N + M]]]), t_obj=env)


def _relv(a, b):
    return float(np.max(np.abs(np.atleast_1d(a) - np.atleast_1d(b))) / max(1.0, np.abs(np.atleast_1d(b)).max()))


def test_host_jvp_matches_the_dense_kkt_solve(host):
    rng = np.random.default_rng(13)
    worst, n = 0.0, 0
    cases = _cases()
    for st, cf, kw in cases[::3] + cases[-4:]:
        r = host.solve(st, cf, **kw)
        p8, m4 = _p8m4(kw)
        u = _tangent(rng, len(cf), p8, m4)
        j = host.jvp(st, cf, r["x"], r["mult"], *u, **kw)
        assert j["status"] == 0
        d = dense_jvp(st, cf, r["x"], r["mult"], u, **kw)
        for k in ("t_traj", "t_out8", "t_obj"):
            worst = max(worst, _relv(j[k], d[k]))
        n += 1
    print(f"host build vs dense KKT solve on {n} problems: max relative difference {worst:.2e}")
    assert worst < 1e-7, worst


def test_host_jvp_matches_finite_differences_of_the_solve(host):
    """Central differences of the host-build solve along random directions (h = 1e-5 of the tangent) within 1e-3
    relative: the problems of the VJP's finite-difference test, and line_params_64 problems at two model rows with active
    steering and acceleration bounds (so d delta_max and d a_max are not trivially zero)."""
    rng = np.random.default_rng(29)
    g = golden("roadmap_256.npz")
    cases = [(g["states"][b], g["fit"][b], {}) for b in (0, 5, 17, 40, 99)]
    cases += [(st, cf, dict(N=LINE_N, ref_v=LINE_REF_V, **_mkw(m4))) for m4 in MODEL_ROWS[:2] for st, cf in _line_problems()[:3]]
    active = np.zeros(2, dtype=int)
    for st, cf, kw in cases:
        r = host.solve(st, cf, **kw)
        p8, m4 = _p8m4(kw)
        N = kw.get("N", 25)
        active += (np.abs(np.abs(r["x"][6 * N:].reshape(2, -1)) - m4[2:, None]) <= 1e-6).sum(1)
        u = _tangent(rng, len(cf), p8 * 0.1, m4 * 0.1)
        j = host.jvp(st, cf, r["x"], r["mult"], *u, **kw)
        h = 1e-5

        def at(a):
            kwa = {**kw, **{k: float(v + a * t) for k, v, t in zip(PNAMES + MNAMES, np.concatenate([p8, m4]),
                                                                    np.concatenate([u[2], u[3]]))}}
            return host.solve(st + a * u[0], np.asarray(cf) + a * u[1], **kwa)
        rp, rm = at(h), at(-h)
        fd_x, fd_obj = (rp["x"] - rm["x"]) / (2 * h), (rp["obj"] - rm["obj"]) / (2 * h)
        assert _relv(j["t_traj"], fd_x) < 1e-3, (kw, _relv(j["t_traj"], fd_x))
        assert _relv(j["t_out8"], (rp["out8"] - rm["out8"]) / (2 * h)) < 1e-3
        assert abs(j["t_obj"] - fd_obj) <= 1e-3 * max(1.0, abs(fd_obj)), (kw, j["t_obj"], fd_obj)
    print(f"stages at an active bound: steering {active[0]}, acceleration {active[1]}")
    assert (active > 0).all(), active


def test_structure_of_the_outputs(host):
    """t_traj's t = 0 states are t_state6 exactly, t_out8 is t_traj's (s_1, delta_0, a_0) bitwise, zero tangents give
    zeros."""
    rng = np.random.default_rng(2)
    N, M = 25, 24
    for st, cf in _problems(4):
        r = host.solve(st, cf)
        p8, m4 = _p8m4({})
        u = _tangent(rng, len(cf), p8, m4)
        j = host.jvp(st, cf, r["x"], r["mult"], *u)
        np.testing.assert_array_equal(j["t_traj"][np.arange(6) * N], u[0])
        np.testing.assert_array_equal(j["t_out8"], np.concatenate([j["t_traj"][np.arange(6) * N + 1],
                                                                   [j["t_traj"][6 * N], j["t_traj"][6 * N + M]]]))
        z = host.jvp(st, cf, r["x"], r["mult"], np.zeros(6), np.zeros(len(cf)), np.zeros(8), np.zeros(4))
        assert z["status"] == 0 and not z["t_traj"].any() and not z["t_out8"].any() and z["t_obj"] == 0.0


def test_failure_statuses(host):
    g = golden("line_256.npz")
    st, cf = g["states"][0], g["coeffs"][0]
    r = host.solve(st, cf)
    ts6 = np.ones(6)
    for bad in ("t_state6", "t_coeffs", "t_cost", "t_model"):
        u = dict(t_state6=ts6, t_coeffs=np.zeros(len(cf)), t_cost=np.zeros(8), t_model=np.zeros(4))
        u[bad] = u[bad].copy()
        u[bad][1] = np.inf if bad == "t_cost" else np.nan
        j = host.jvp(st, cf, r["x"], r["mult"], **u)
        assert j["status"] == -13 and np.isnan(j["t_traj"]).all() and np.isnan(j["t_out8"]).all() and np.isnan(j["t_obj"])
    # a negative bound multiplier, as test_sensitivity.test_failure_statuses: the control block of the factor is
    # indefinite there
    m = r["mult"].copy()
    m[150 + 3] = -1e9
    j = host.jvp(st, cf, r["x"], m, ts6)
    assert j["status"] == -3 and np.isnan(j["t_traj"]).all() and np.isnan(j["t_obj"])


def test_argument_errors_of_the_jvp_entries_do_not_need_a_gpu():
    import udacitympc_b200 as mp
    lib = mp.load_library()
    err = lambda: lib.b200mpc_last_error()
    P = _p(np.zeros(64))
    fake = ctypes.create_string_buffer(1 << 16)   # every call below fails its argument check before the handle is read
    h = ctypes.cast(fake, ctypes.c_void_p)
    jvp, jvpd = lib.b200mpc_solve_batch_jvp, lib.b200mpc_solve_batch_jvp_device
    assert jvp(None, 1, P, P, 4, None, None, P, P, P, None, None, None, P, None, None, None) == -1
    assert b"null handle" in err()
    assert jvp(h, 0, P, P, 4, None, None, P, P, P, None, None, None, P, None, None, None) == -1
    assert b"B must be positive" in err()
    assert jvp(h, 1, P, P, 5, None, None, P, P, P, None, None, None, P, None, None, None) == -1
    assert b"ncoef" in err()
    assert jvp(h, 1, P, P, 4, None, None, None, P, P, None, None, None, P, None, None, None) == -1
    assert b"null state6 / coeffs / traj / mult" in err()
    assert jvp(h, 1, P, P, 4, None, None, P, P, None, None, None, None, P, None, None, None) == -1
    assert b"no tangent" in err()
    assert jvpd(None, 1, 1, 1, 4, None, None, 1, 1, 1, None, None, None, 1, None, None, None, None) == -1
    assert b"null handle" in err()
    assert jvpd(h, -1, 1, 1, 4, None, None, 1, 1, 1, None, None, None, 1, None, None, None, None) == -1
    assert b"B must be positive" in err()
    assert jvpd(h, 1, 1, 1, 1, None, None, 1, 1, 1, None, None, None, 1, None, None, None, None) == -1
    assert b"ncoef" in err()
    assert jvpd(h, 1, 1, None, 4, None, None, 1, 1, 1, None, None, None, 1, None, None, None, None) == -1
    assert b"null state6 / coeffs / traj / mult" in err()
    assert jvpd(h, 1, 1, 1, 4, 1, 1, 1, 1, None, None, None, None, 1, None, None, None, None) == -1
    assert b"no tangent" in err()


def test_shape_errors_of_the_python_wrapper():
    """Shapes are checked before any library call (so without a GPU)."""
    import udacitympc_b200 as mp
    stub = types.SimpleNamespace(num_vars=198, num_mults=246, _lib=None, _h=None)
    call = lambda **kw: mp.MPC.solve_batch_jvp(stub, **{**dict(states=np.zeros((3, 6)), coeffs=np.zeros(4),
                                                                 traj=np.zeros((3, 198)), mult=np.zeros((3, 246))), **kw})
    for kw in (dict(states=np.zeros((3, 5))), dict(coeffs=np.zeros((2, 4))), dict(traj=np.zeros((3, 197))),
               dict(t_state6=np.zeros(6)), dict(t_coeffs=np.zeros(3)), dict(t_coeffs=np.zeros((2, 4))),
               dict(t_cost=np.zeros(7)), dict(t_model=np.zeros((3, 5))), dict(cost_params=np.zeros((2, 8)))):
        with pytest.raises(ValueError):
            call(**kw)


def test_header_declares_the_jvp_entries():
    from udacitympc_b200 import api
    with open(os.path.join(ROOT, "include", "b200mpc.h")) as f:
        text = f.read()
    for name in ("b200mpc_solve_batch_jvp", "b200mpc_solve_batch_jvp_device"):
        assert name in api.SYMBOLS and f"int {name}(" in text


# ------------------------------------------------------------------------------------------------ GPU
gpu = pytest.mark.skipif(not has_gpu(), reason="needs a CUDA device")


def _bench():
    sys.path.insert(0, ROOT)
    import bench
    return bench


def _dev(a):
    import torch
    return torch.as_tensor(np.ascontiguousarray(np.asarray(a, dtype=np.float64).T), device="cuda")


def _rand_tangents(rng, B, ncoef, p8, m4):
    return (rng.standard_normal((B, 6)), rng.standard_normal((B, ncoef)) * CF_SCALE[:ncoef],
            rng.standard_normal((B, 8)) * p8, rng.standard_normal((B, 4)) * m4)


@pytest.mark.gpu
@gpu
@pytest.mark.parametrize("name,N", [("roadmap_256.npz", 25), ("roadmap_N10_64.npz", 10), ("roadmap_N50_64.npz", 50),
                                    ("roadmap_N100_64.npz", 100)])
def test_device_jvp_matches_the_host_build(host, name, N):
    import udacitympc_b200 as mp
    g = golden(name)
    st, cf = g["states"], _coeffs(g)
    rng = np.random.default_rng(N)
    p8, m4 = _p8m4(dict(N=N))
    u = _rand_tangents(rng, len(st), cf.shape[1], p8, m4)
    with mp.MPC(N=N) as mpc:
        r = mpc.solve_batch(st, cf, want_traj=True, want_mult=True)
        j = mpc.solve_batch_jvp(st, cf, r["traj"], r["mult"], *u)
    worst, n = 0.0, 0
    for b in range(len(st)):
        if r["status"][b] not in (0, 1):
            continue
        h = host.jvp(st[b], cf[b], r["traj"][b], r["mult"][b], *[t[b] for t in u], N=N)
        assert j["status"][b] == h["status"] == 0, b
        for k in ("t_out8", "t_traj", "t_obj"):
            worst = max(worst, _relv(j[k][b], h[k]))
        n += 1
    assert n >= len(st) // 2
    print(f"device vs host build, {name}: max relative difference {worst:.2e} over {n} problems")
    assert worst < 1e-10, worst


@pytest.mark.gpu
@gpu
def test_device_jvp_with_random_rows_matches_the_host_build(host):
    """4 096 bench problems at N = 25 with random cost and model rows; a sample of 256 of those whose iteration counts
    match the host build's solve."""
    import udacitympc_b200 as mp
    rng = np.random.default_rng(41)
    B = 4096
    with mp.MPC() as mpc:
        st, cf = _bench().make_workload("roadmap", B, mpc=mpc)
        c8, m4 = _random_costs(rng, B), _random_models(rng, B)
        r = mpc.solve_batch(st, cf, want_traj=True, want_mult=True, cost_params=c8, model_params=m4)
        u = _rand_tangents(rng, B, cf.shape[1], c8, m4)
        j = mpc.solve_batch_jvp(st, cf, r["traj"], r["mult"], *u, cost_params=c8, model_params=m4)
    worst, n = 0.0, 0
    for b in rng.permutation(np.flatnonzero(r["status"] == 0)):
        kw = {**_kw(c8[b]), **_mkw(m4[b])}
        hs = host.solve(st[b], cf[b], **kw)
        if hs["iters"] != r["iters"][b]:
            continue
        h = host.jvp(st[b], cf[b], r["traj"][b], r["mult"][b], *[t[b] for t in u], **kw)
        assert j["status"][b] == h["status"] == 0
        for k in ("t_out8", "t_traj", "t_obj"):
            worst = max(worst, _relv(j[k][b], h[k]))
        n += 1
        if n == 256:
            break
    assert n == 256
    print(f"device vs host build, random cost and model rows: max relative difference {worst:.2e} over {n} problems")
    assert worst < 1e-10, worst


@pytest.mark.gpu
@gpu
def test_adjoint_identity_on_the_bench_workload():
    """All 65 536 problems of the benchmark's workload at N = 25: the device JVP along random tangents of all four groups
    against the device VJP along random cotangents."""
    import udacitympc_b200 as mp
    rng = np.random.default_rng(43)
    B = 65536
    with mp.MPC() as mpc:
        st, cf = _bench().make_workload("roadmap", B, mpc=mpc)
        r = mpc.solve_batch(st, cf, want_traj=True, want_mult=True)
        p8, m4 = _p8m4({})
        u = _rand_tangents(rng, B, cf.shape[1], p8, m4)
        go8, gt, gob = rng.standard_normal((B, 8)), rng.standard_normal((B, mpc.num_vars)), rng.standard_normal(B)
        j = mpc.solve_batch_jvp(st, cf, r["traj"], r["mult"], *u)
        v = mpc.solve_batch_vjp(st, cf, r["traj"], r["mult"], go8, gt, gob, want_params=True, want_model=True)
    conv = (r["status"] == 0) | (r["status"] == 1)
    assert conv.mean() > 0.99
    assert (j["status"][conv] == 0).all() and (v["status"][conv] == 0).all()
    lhs = np.concatenate([go8 * j["t_out8"], gt * j["t_traj"], (gob * j["t_obj"])[:, None]], axis=1)[conv]
    rhs = np.concatenate([v[k] * t for k, t in zip(("grad_state6", "grad_coeffs", "grad_params", "grad_model"), u)],
                         axis=1)[conv]
    d = np.abs(lhs.sum(1) - rhs.sum(1)) / (np.abs(lhs).sum(1) + np.abs(rhs).sum(1))
    print(f"adjoint identity on the device, {conv.sum()} problems: max {d.max():.2e}")
    assert d.max() <= 1e-10, d.max()


@pytest.mark.gpu
@gpu
def test_host_and_device_entries_agree_bitwise_and_launch_once():
    import torch
    import udacitympc_b200 as mp
    g = golden("roadmap_256.npz")
    st, cf = g["states"], g["fit"]
    rng = np.random.default_rng(1)
    with mp.MPC() as mpc:
        c8, m4 = _random_costs(rng, 256), _random_models(rng, 256)
        r = mpc.solve_batch(st, cf, want_traj=True, want_mult=True, cost_params=c8, model_params=m4)
        u = _rand_tangents(rng, 256, 4, c8, m4)
        for rows in ((None, None), (c8, None), (c8, m4)):
            for tg in (u, (u[0], u[1], u[2], None)):
                j = mpc.solve_batch_jvp(st, cf, r["traj"], r["mult"], *tg, cost_params=rows[0], model_params=rows[1])
                ins = [_dev(st), _dev(cf)] + [None if a is None else _dev(a) for a in rows] + [_dev(r["traj"]), _dev(r["mult"])]
                ins += [None if a is None else _dev(a) for a in tg]
                E = lambda *s: torch.empty(s, dtype=torch.float64, device="cuda")
                to8, tt, tob = E(8, 256), E(mpc.num_vars, 256), E(256)
                vs = torch.empty(256, dtype=torch.int32, device="cuda")
                torch.cuda.synchronize()   # the call below runs on the handle's own stream
                n0 = mpc.launch_count()
                ptr = lambda a: 0 if a is None else a.data_ptr()
                mpc.solve_batch_jvp_device(256, ptr(ins[0]), ptr(ins[1]), 4, *[ptr(a) for a in ins[2:]], to8.data_ptr(),
                                           tt.data_ptr(), tob.data_ptr(), vs.data_ptr())
                mpc.wait()
                assert mpc.launch_count() == n0 + 1
                np.testing.assert_array_equal(to8.cpu().numpy().T, j["t_out8"])
                np.testing.assert_array_equal(tt.cpu().numpy().T, j["t_traj"])
                np.testing.assert_array_equal(tob.cpu().numpy(), j["t_obj"])
                np.testing.assert_array_equal(vs.cpu().numpy(), j["status"])


@pytest.mark.gpu
@gpu
def test_invalid_rows_and_tangents_and_graph_capture():
    """A non-finite tangent, cost row or model row gives that problem -13 and NaN outputs and leaves its neighbours as
    they are; the device entry can be captured into a CUDA graph once the workspace has grown."""
    import torch
    import udacitympc_b200 as mp
    g = golden("roadmap_256.npz")
    st, cf = g["states"][:64], g["fit"][:64]
    rng = np.random.default_rng(3)
    with mp.MPC() as mpc:
        r = mpc.solve_batch(st, cf, want_traj=True, want_mult=True)
        p8, m4 = _p8m4({})
        u = _rand_tangents(rng, 64, 4, p8, m4)
        want = mpc.solve_batch_jvp(st, cf, r["traj"], r["mult"], *u, cost_params=p8, model_params=m4)
        bad_u = [a.copy() for a in u]
        bad_u[0][3, 2] = np.nan
        bad_u[3][5, 0] = np.inf
        c8b, m4b = np.tile(p8, (64, 1)), np.tile(m4, (64, 1))
        c8b[7, 1] = np.nan
        m4b[9, 1] = -1.0
        got = mpc.solve_batch_jvp(st, cf, r["traj"], r["mult"], *bad_u, cost_params=c8b, model_params=m4b)
        badset = [3, 5, 7, 9]
        ok = np.setdiff1d(np.arange(64), badset)
        assert (got["status"][badset] == -13).all()
        for k in ("t_out8", "t_traj", "t_obj"):
            assert np.isnan(got[k][badset]).all()
            np.testing.assert_array_equal(got[k][ok], want[k][ok])
        np.testing.assert_array_equal(got["status"][ok], want["status"][ok])
        # graph capture on a pre-grown workspace
        ins = [_dev(st), _dev(cf), _dev(r["traj"]), _dev(r["mult"]), _dev(u[0]), _dev(u[1])]
        E = lambda *s: torch.empty(s, dtype=torch.float64, device="cuda")
        to8, tt, tob = E(8, 64), E(mpc.num_vars, 64), E(64)
        s = torch.cuda.Stream()
        graph = torch.cuda.CUDAGraph()
        torch.cuda.synchronize()
        with torch.cuda.graph(graph, stream=s):
            mpc.solve_batch_jvp_device(64, ins[0].data_ptr(), ins[1].data_ptr(), 4, 0, 0, ins[2].data_ptr(), ins[3].data_ptr(),
                                       ins[4].data_ptr(), ins[5].data_ptr(), 0, 0, to8.data_ptr(), tt.data_ptr(),
                                       tob.data_ptr(), 0, stream=s.cuda_stream)
        graph.replay()
        torch.cuda.synchronize()
        j = mpc.solve_batch_jvp(st, cf, r["traj"], r["mult"], u[0], u[1])
        np.testing.assert_array_equal(to8.cpu().numpy().T, j["t_out8"])
        np.testing.assert_array_equal(tt.cpu().numpy().T, j["t_traj"])
        np.testing.assert_array_equal(tob.cpu().numpy(), j["t_obj"])


@pytest.mark.gpu
@gpu
def test_jvp_after_pipelined_solves_equals_a_plain_handle():
    import torch
    import udacitympc_b200 as mp
    g = golden("roadmap_256.npz")
    st, cf = g["states"], g["fit"]
    rng = np.random.default_rng(9)
    with mp.MPC() as plain:
        r = plain.solve_batch(st, cf, want_traj=True, want_mult=True)
        ts6, tcf = rng.standard_normal((256, 6)), rng.standard_normal((256, 4)) * CF_SCALE
        want = plain.solve_batch_jvp(st, cf, r["traj"], r["mult"], ts6, tcf)
    with mp.MPC() as mpc:
        mpc.set_pipeline(4, 1024)
        B = 16384
        bs, bc = _bench().make_workload("roadmap", B, mpc=mpc)
        d_st, d_cf = _dev(bs), _dev(bc)
        streams = [torch.cuda.Stream() for _ in range(3)]
        torch.cuda.synchronize()
        outs = []
        for s in streams:
            o = torch.empty(8, B, dtype=torch.float64, device="cuda")
            outs.append(o)
            mpc.solve_batch_device(B, d_st.data_ptr(), d_cf.data_ptr(), 4, o.data_ptr(), stream=s.cuda_stream)
        got = mpc.solve_batch_jvp(st, cf, r["traj"], r["mult"], ts6, tcf)
        torch.cuda.synchronize()
    for k in ("t_out8", "t_traj", "t_obj", "status"):
        np.testing.assert_array_equal(got[k], want[k])


@pytest.mark.gpu
@gpu
@pytest.mark.parametrize("where", ["cuda", "cpu"])
@pytest.mark.parametrize("shared", [False, True])
def test_forward_ad_equals_the_direct_jvp_and_the_backward_pass(where, shared):
    """torch.autograd.forward_ad through autograd.solve: the tangents equal MPC.solve_batch_jvp's (tangents of shared
    inputs apply to every problem), and <cotangent, forward tangent> equals <backward gradient, tangent>."""
    import torch
    import torch.autograd.forward_ad as fwAD
    import udacitympc_b200 as mp
    from udacitympc_b200 import autograd
    g = golden("roadmap_256.npz")
    B = 128
    st_np, cf_np = g["states"][:B], (g["fit"][3] if shared else g["fit"][:B])
    rng = np.random.default_rng(4)
    p8, m4 = _p8m4({})
    c8_np, m4_np = (p8, m4) if shared else (np.tile(p8, (B, 1)), np.tile(m4, (B, 1)))
    ncoef = 4
    tangents = [rng.standard_normal((B, 6)), rng.standard_normal(cf_np.shape) * CF_SCALE,
                rng.standard_normal(c8_np.shape) * p8, rng.standard_normal(m4_np.shape) * m4]
    T = lambda a: torch.tensor(a, device=where)
    with mp.MPC() as mpc:
        with fwAD.dual_level():
            duals = [fwAD.make_dual(T(a), T(t)) for a, t in zip((st_np, cf_np, c8_np, m4_np), tangents)]
            out8, traj, obj, status = autograd.solve(mpc, *duals[:2], cost_params=duals[2], model_params=duals[3])
            t8, tt, to = (fwAD.unpack_dual(o).tangent for o in (out8, traj, obj))
        r = mpc.solve_batch(st_np, cf_np, want_traj=True, want_mult=True, cost_params=c8_np, model_params=m4_np)
        bt = [np.broadcast_to(t, s) for t, s in zip(tangents, ((B, 6), (B, ncoef), (B, 8), (B, 4)))]
        j = mpc.solve_batch_jvp(st_np, cf_np, r["traj"], r["mult"], *bt, cost_params=c8_np, model_params=m4_np)
        assert (status.cpu().numpy() == 0).all()
        np.testing.assert_array_equal(t8.cpu().numpy(), j["t_out8"])
        np.testing.assert_array_equal(tt.cpu().numpy(), j["t_traj"])
        np.testing.assert_array_equal(to.cpu().numpy(), j["t_obj"])
        # the backward pass of the same function: <w, J u> = <J^T w, u>
        leaves = [T(a).requires_grad_() for a in (st_np, cf_np, c8_np, m4_np)]
        o8, otr, oo, _ = autograd.solve(mpc, *leaves[:2], cost_params=leaves[2], model_params=leaves[3])
        w8, wt, wo = (rng.standard_normal(s) for s in ((B, 8), (B, mpc.num_vars), (B,)))
        loss = (o8 * T(w8)).sum() + (otr * T(wt)).sum() + (oo * T(wo)).sum()
        grads = torch.autograd.grad(loss, leaves)
    lhs = (w8 * t8.cpu().numpy()).sum() + (wt * tt.cpu().numpy()).sum() + (wo * to.cpu().numpy()).sum()
    terms = [(gr.cpu().numpy() * t) for gr, t in zip(grads, tangents)]
    rhs = sum(x.sum() for x in terms)
    scale = np.abs(w8 * t8.cpu().numpy()).sum() + np.abs(wt * tt.cpu().numpy()).sum() + sum(np.abs(x).sum() for x in terms)
    assert abs(lhs - rhs) <= 1e-10 * scale, (lhs, rhs, scale)
