"""Warm start from a caller-supplied primal-dual point and the returned multipliers (b200mpc_solve_batch_warm, not
reference behaviour).  CPU tests run the host build of the solver core (tests/hostsim/hostsim_guess.cpp) in three
execution shapes; -m gpu runs the same checks through the C ABI on every launch schedule."""
import ctypes

import numpy as np
import pytest

from conftest import golden

dp = ctypes.POINTER(ctypes.c_double)
ip = ctypes.POINTER(ctypes.c_int)
MODES = {"trip": 0, "per_pass_repacked": -2, "coop": 2}


def _p(a):
    return None if a is None else a.ctypes.data_as(dp)


def _nm(N):
    return 10 * N - 4


def shift(traj, mult, N):
    import udacitympc_b200 as mp
    return mp.shift_solution(traj, mult, N)


@pytest.fixture(scope="module")
def guess(_build_everything):
    """hostsim_solve_guess (tests/hostsim/hostsim_guess.cpp): one solve from (x_init, mult_init) -- x_init None: the
    default start -- in an execution mode."""
    import os
    import oracle_bindings as ob
    lib = ctypes.CDLL(os.path.join(ob.ROOT, "tests", "hostsim", "libhostsim_guess.so"))

    def solve(state6, coeffs, x_init=None, mult_init=None, mu_init=1e-4, mode="trip", **params):
        p = ob.default_params(**params)
        N = p.N
        st = np.ascontiguousarray(state6, dtype=np.float64); c = np.ascontiguousarray(coeffs, dtype=np.float64)
        xi = None if x_init is None else np.ascontiguousarray(x_init, dtype=np.float64)
        mi = None if mult_init is None else np.ascontiguousarray(mult_init, dtype=np.float64)
        x = np.zeros(8 * N - 2); o8 = np.zeros(8); obj = ctypes.c_double(); it = ctypes.c_int(); m = np.zeros(_nm(N))
        rc = lib.hostsim_solve_guess(ctypes.byref(p), _p(st), _p(c), len(c), _p(xi), _p(mi), ctypes.c_double(mu_init),
                                             _p(x), _p(o8), ctypes.byref(obj), ctypes.byref(it), _p(m), MODES[mode])
        return dict(status=rc, x=x, out8=o8, obj=obj.value, iters=it.value, mult=m)
    return solve


def kkt_residual(x, mult, coeffs, N):
    """grad f + J^T lambda - z_L + z_U at x, by the C port's own evaluator (unscaled problem), and the complementarity
    products z * slack of the control bounds."""
    import oracle_bindings as ob
    p = ob.default_params(N=N)
    M = N - 1
    lam = mult[:6 * N]
    _, grad, _, J, _ = ob.port_eval(x, lam, coeffs, params=p)
    zl = np.zeros(8 * N - 2); zu = np.zeros(8 * N - 2)
    zl[6 * N:] = mult[6 * N:6 * N + 2 * M]; zu[6 * N:] = mult[6 * N + 2 * M:]
    r = grad + J.T @ lam - zl + zu
    bnd = np.concatenate([np.full(M, p.delta_max), np.full(M, p.a_max)])
    u = x[6 * N:]
    comp = np.concatenate([zl[6 * N:] * (u + bnd), zu[6 * N:] * (bnd - u)])
    return r[6:], comp   # the rows of s_0 are fixed by the initial-state constraints (their lambda takes any residual)


# ------------------------------------------------------------------------------------------------ CPU (host build)
@pytest.mark.parametrize("name", ["line_256.npz", "roadmap_256.npz"])
def test_cold_multipliers_match_the_oracle(guess, name):
    import oracle_bindings as ob
    g = golden(name)
    cf = g["coeffs"] if "coeffs" in g.files else g["fit"]
    for b in range(0, 256, 16):
        r = guess(g["states"][b], cf[b])
        o = ob.port_solve(g["states"][b], cf[b])
        if r["status"] != 0 or r["iters"] != o["iters"]:
            continue
        scale = max(1.0, np.abs(o["lam"]).max())
        np.testing.assert_allclose(r["mult"][:150], o["lam"], rtol=0, atol=1e-9 * scale)
        res, comp = kkt_residual(r["x"], r["mult"], cf[b], 25)
        assert np.abs(res).max() <= 1e-6 * scale, (b, np.abs(res).max())
        assert (r["mult"][150:] > 0).all() and np.abs(comp).max() < 1e-6
        if ob.ref_available():
            rf = ob.ref_solve(g["states"][b], cf[b])
            np.testing.assert_allclose(r["mult"][:150], rf["lam"], rtol=0, atol=1e-6 * scale)
            np.testing.assert_allclose(r["mult"][150:198], rf["zl"][150:], rtol=0, atol=1e-6)
            np.testing.assert_allclose(r["mult"][198:], rf["zu"][150:], rtol=0, atol=1e-6)


def test_receding_horizon_from_the_shifted_solution(guess):
    """config 1's 50-step closed loop: step k+1 starts from step k's solution and multipliers shifted by one stage
    (observed: 272 iterations instead of the cold 739)."""
    g = golden("config1_closed_loop.npz")
    r = guess(g["states"][0], g["coeffs"])
    total = r["iters"]
    for k in range(1, 50):
        x0, m0 = shift(r["x"], r["mult"], 25)
        r = guess(g["states"][k], g["coeffs"], x0, m0)
        assert r["status"] == 0
        np.testing.assert_allclose(r["out8"], g["out8"][k], rtol=0, atol=1e-7)
        total += r["iters"]
    assert total < 0.5 * g["iters"].sum(), (total, g["iters"].sum())


def test_start_at_the_optimum(guess):
    """From a problem's own solution and multipliers: the same solution in fewer iterations.  Observed on these 16
    problems: 227 iterations cold, 61 warm (3 to 7 each; problem 0: 17 -> 5)."""
    g = golden("line_256.npz")
    cold = warm = 0
    for b in range(16):
        c = guess(g["states"][b], g["coeffs"][b])
        w = guess(g["states"][b], g["coeffs"][b], c["x"], c["mult"])
        assert w["status"] == c["status"] == 0
        assert w["iters"] < c["iters"], b
        np.testing.assert_allclose(w["out8"], c["out8"], rtol=0, atol=1e-7)
        cold += c["iters"]; warm += w["iters"]
    assert warm < 0.5 * cold, (warm, cold)


@pytest.mark.parametrize("with_mult", [True, False])
def test_execution_modes_agree(guess, with_mult):
    g = golden("roadmap_256.npz")
    for b in (1, 7, 42):
        c = guess(g["states"][b], g["fit"][b])
        x0, m0 = shift(c["x"], c["mult"], 25)
        st = g["states"][b].copy(); st[3] += 0.5   # a different initial state: not at the optimum
        rs = [guess(st, g["fit"][b], x0, m0 if with_mult else None, mode=m) for m in MODES]
        for r in rs[1:]:
            assert r["status"] == rs[0]["status"] and r["iters"] == rs[0]["iters"]
            np.testing.assert_allclose(r["x"], rs[0]["x"], rtol=0, atol=1e-10)
            np.testing.assert_allclose(r["mult"], rs[0]["mult"], rtol=0, atol=1e-10 * max(1.0, np.abs(rs[0]["mult"]).max()))


@pytest.mark.parametrize("mode", sorted(MODES))
def test_invalid_guess(guess, mode):
    g = golden("line_256.npz")
    c = guess(g["states"][0], g["coeffs"][0])
    for where in ("x", "mult"):
        x0, m0 = c["x"].copy(), c["mult"].copy()
        (x0 if where == "x" else m0)[60] = np.nan
        r = guess(g["states"][0], g["coeffs"][0], x0, m0, mode=mode)
        assert r["status"] == -13 and r["iters"] == 0


def test_shift_solution_layouts():
    import udacitympc_b200 as mp
    N, B = 5, 3
    rng = np.random.default_rng(0)
    x = rng.normal(size=(B, 8 * N - 2)); m = rng.normal(size=(B, _nm(N)))
    xs, ms = mp.shift_solution(x, m, N)
    st = x[:, :6 * N].reshape(B, 6, N)
    np.testing.assert_array_equal(xs[:, :6 * N].reshape(B, 6, N)[:, :, :-1], st[:, :, 1:])
    np.testing.assert_array_equal(xs[:, :6 * N].reshape(B, 6, N)[:, :, -1], st[:, :, -1])
    u = x[:, 6 * N:].reshape(B, 2, N - 1)
    np.testing.assert_array_equal(xs[:, 6 * N:].reshape(B, 2, N - 1)[:, :, :-1], u[:, :, 1:])
    z = m[:, 6 * N:].reshape(B, 4, N - 1)
    np.testing.assert_array_equal(ms[:, 6 * N:].reshape(B, 4, N - 1)[:, :, :-1], z[:, :, 1:])
    np.testing.assert_array_equal(ms[:, 6 * N:].reshape(B, 4, N - 1)[:, :, -1], z[:, :, -1])
    xf, mf = mp.shift_solution(x.T.copy(), m.T.copy(), N)   # field-major
    np.testing.assert_array_equal(xf, xs.T); np.testing.assert_array_equal(mf, ms.T)
    assert mp.shift_solution(x, None, N)[1] is None
    torch = pytest.importorskip("torch")
    xt, mt = mp.shift_solution(torch.from_numpy(x.T.copy()), torch.from_numpy(m.T.copy()), N, field_major=True)
    np.testing.assert_array_equal(xt.numpy(), xs.T); np.testing.assert_array_equal(mt.numpy(), ms.T)
    with pytest.raises(ValueError):
        mp.shift_solution(np.zeros((8 * N - 2, 8 * N - 2)), None, N)


# ------------------------------------------------------------------------------------------------ GPU (C ABI)
def _roadmap(B, N=25):
    from udacitympc_b200 import synth
    if N == 25:
        g = golden("roadmap_256.npz")
        idx = np.arange(B) % 256
        return np.ascontiguousarray(g["states"][idx]), np.ascontiguousarray(g["fit"][idx])
    g = golden(f"roadmap_N{N}_64.npz")
    idx = np.arange(B) % 64
    return np.ascontiguousarray(g["states"][idx]), np.ascontiguousarray(g["coeffs"][idx])


def _mpc(N=25, **settings):
    import udacitympc_b200 as mp
    m = mp.MPC(device=0, N=N, max_iter=3000 if N <= 100 else 400)
    for name, args in settings.items():
        getattr(m, name)(*args)
    return m


def _check_warm_call(m, st, cf, N):
    """cold with multipliers, then a warm start at the optimum and from a perturbed state: what every schedule must do"""
    c = m.solve_batch(st, cf, want_traj=True, want_mult=True)
    ok = c["status"] == 0
    assert ok.mean() > 0.9
    w = m.solve_batch(st, cf, want_traj=True, x_init=c["traj"], mult_init=c["mult"], want_mult=True)
    assert (w["status"][ok] == 0).all()
    np.testing.assert_allclose(w["out8"][ok], c["out8"][ok], rtol=0, atol=1e-6)   # same local optimum within the tolerance
    assert w["iters"][ok].sum() < 0.6 * c["iters"][ok].sum(), (w["iters"][ok].sum(), c["iters"][ok].sum())
    for b in np.flatnonzero(ok)[:4]:   # the returned multipliers satisfy the KKT conditions
        res, comp = kkt_residual(w["traj"][b], w["mult"][b], cf[b], N)
        scale = max(1.0, np.abs(w["mult"][b][:6 * N]).max())
        assert np.abs(res).max() <= 1e-6 * scale and np.abs(comp).max() < 1e-6
    return c, w


@pytest.mark.gpu
@pytest.mark.parametrize("B", [100, 4096, 16384])
def test_gpu_warm_start(guess, B):
    """latency path (100: cooperative kernel) and throughput path (compaction, split 4); hostsim agrees on a sample"""
    st, cf = _roadmap(B)
    with _mpc() as m:
        c, w = _check_warm_call(m, st, cf, 25)
        for b in (0, 3, 77):
            o = guess(st[b], cf[b])
            assert o["iters"] == c["iters"][b]
            np.testing.assert_allclose(c["mult"][b][:150], o["mult"][:150], rtol=0, atol=1e-7 * max(1.0, np.abs(o["mult"]).max()))
            h = guess(st[b], cf[b], c["traj"][b], c["mult"][b])
            assert h["iters"] == w["iters"][b]


@pytest.mark.gpu
def test_gpu_warm_start_fused():
    st, cf = _roadmap(4096)
    with _mpc(set_solver_mode=(1, 0, -1)) as m:
        _check_warm_call(m, st, cf, 25)


@pytest.mark.gpu
@pytest.mark.parametrize("N,B", [(10, 4096), (50, 4096), (100, 512), (200, 40)])
def test_gpu_warm_start_horizons(N, B):
    """N = 200: the cooperative kernel with one problem per block starts from the guess"""
    if N == 200:
        from udacitympc_b200 import synth
        st, cf = synth.line_problems(B)
    else:
        st, cf = _roadmap(B, N)
    with _mpc(N=N) as m:
        _check_warm_call(m, st, cf, N)


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 4096])
def test_gpu_receding_horizon(B):
    """config 1's closed loop through the C ABI, every step warm-started from the previous one shifted"""
    import udacitympc_b200 as mp
    g = golden("config1_closed_loop.npz")
    cf = np.tile(g["coeffs"], (B, 1))
    with _mpc() as m:
        r = m.solve_batch(np.tile(g["states"][0], (B, 1)), cf, want_traj=True, want_mult=True)
        total = r["iters"].astype(np.int64)
        for k in range(1, 50):
            x0, m0 = mp.shift_solution(r["traj"], r["mult"], 25)
            r = m.solve_batch(np.tile(g["states"][k], (B, 1)), cf, want_traj=True, x_init=x0, mult_init=m0, want_mult=True)
            assert (r["status"] == 0).all()
            np.testing.assert_allclose(r["out8"], np.tile(g["out8"][k], (B, 1)), rtol=0, atol=1e-7)
            total += r["iters"]
        assert (total < 0.5 * g["iters"].sum()).all()


@pytest.mark.gpu
def test_gpu_pipelined_warm_start():
    st, cf = _roadmap(16384)
    with _mpc() as m:
        c = m.solve_batch(st, cf, want_traj=True, want_mult=True)
        x0, m0 = shift(c["traj"], c["mult"], 25)
        st2 = st.copy(); st2[:, 3] += 0.3
        plain = m.solve_batch(st2, cf, want_traj=True, x_init=x0, mult_init=m0, want_mult=True)
    with _mpc(set_pipeline=(2, 1024)) as m:
        for _ in range(2):
            p = m.solve_batch(st2, cf, want_traj=True, x_init=x0, mult_init=m0, want_mult=True)
            np.testing.assert_array_equal(p["status"], plain["status"])
            np.testing.assert_array_equal(p["iters"], plain["iters"])
            for k in ("out8", "traj", "mult"):
                np.testing.assert_allclose(p[k], plain[k], rtol=0, atol=1e-9 * max(1.0, np.abs(plain[k]).max()))


@pytest.mark.gpu
@pytest.mark.parametrize("B", [100, 4096])
def test_gpu_cold_through_the_warm_entry_is_bitwise_the_plain_solve(B):
    st, cf = _roadmap(B)
    with _mpc() as m:
        a = m.solve_batch(st, cf, want_traj=True)
        b = m.solve_batch(st, cf, want_traj=True, want_mult=True)
        for k in ("out8", "cost", "status", "iters", "traj"):
            np.testing.assert_array_equal(a[k], b[k])
        assert np.isfinite(b["mult"]).all()


@pytest.mark.gpu
def test_gpu_graph_key_covers_the_guess():
    """Two calls on one handle that differ only in mu_init or in the guess buffer return what fresh handles return
    (a replayed graph with the first call's arguments would not)."""
    torch = pytest.importorskip("torch")
    st, cf = _roadmap(4096)
    with _mpc() as m0:
        c = m0.solve_batch(st, cf, want_traj=True, want_mult=True)
    x0, mu0 = shift(c["traj"], c["mult"], 25)
    dev = torch.device("cuda:0")
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a.T)).to(dev)
    dst, dcf = T(st), T(cf)
    g1x, g1m = T(c["traj"]), T(c["mult"])
    g2x, g2m = T(x0), T(mu0)
    torch.cuda.synchronize()   # the solves run on the handle's own stream

    def call(m, gx, gm, mu):
        out = torch.empty((8, 4096), dtype=torch.float64, device=dev); it = torch.empty(4096, dtype=torch.int32, device=dev)
        m.solve_batch_warm_device(4096, dst.data_ptr(), dcf.data_ptr(), 4, gx.data_ptr(), gm.data_ptr(), mu, out.data_ptr(),
                                  d_iters=it.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        return out.cpu().numpy(), it.cpu().numpy()

    with _mpc() as m:
        seq = [call(m, g1x, g1m, 1e-4), call(m, g1x, g1m, 1e-2), call(m, g2x, g2m, 1e-4)]
    for (gx, gm, mu), got in zip([(g1x, g1m, 1e-4), (g1x, g1m, 1e-2), (g2x, g2m, 1e-4)], seq):
        with _mpc() as f:
            ref = call(f, gx, gm, mu)
        np.testing.assert_array_equal(got[0], ref[0]); np.testing.assert_array_equal(got[1], ref[1])
    assert not np.array_equal(seq[0][1], seq[1][1]) or not np.array_equal(seq[0][0], seq[1][0])


@pytest.mark.gpu
@pytest.mark.parametrize("launches", ["graphs", "plain"])
def test_gpu_warm_launch_counts(launches, monkeypatch):
    """84 launches as a cold solve at B = 4096, plus one transpose each for x_init, mult_init, mult (and traj)"""
    monkeypatch.setenv("B200MPC_NO_GRAPHS", "1" if launches == "plain" else "0")
    st, cf = _roadmap(4096)
    with _mpc() as m:
        c = m.solve_batch(st, cf, want_traj=True, want_mult=True)
        for kw, expected in [(dict(want_mult=True), 85), (dict(x_init=c["traj"]), 85),
                             (dict(x_init=c["traj"], mult_init=c["mult"], want_mult=True), 87),
                             (dict(x_init=c["traj"], mult_init=c["mult"], want_mult=True, want_traj=True), 88)]:
            for _ in range(2):   # capture, replay
                n = m.launch_count()
                m.solve_batch(st, cf, **kw)
                assert m.launch_count() - n == expected, kw


@pytest.mark.gpu
def test_gpu_argument_errors():
    import udacitympc_b200 as mp
    st, cf = _roadmap(8)
    with _mpc() as m:
        x = np.zeros((8, m.num_vars)); mu = np.zeros((8, m.num_mults))
        assert m.num_mults == 246
        for kw in [dict(x_init=x, mu_init=0.0), dict(x_init=x, mu_init=0.2), dict(x_init=x, mu_init=float("nan")),
                   dict(mult_init=mu)]:
            with pytest.raises(mp.B200MPCError):
                m.solve_batch(st, cf, **kw)
        with pytest.raises(ValueError):
            m.solve_batch(st, cf, x_init=np.zeros((8, 5)))
        r = m.solve_batch(st, cf, x_init=x, mu_init=0.1)   # the bounds themselves are valid
        assert r["status"].shape == (8,)
        c = m.solve_batch(st, cf, want_traj=True)
        xb = c["traj"].copy(); xb[3, 101] = np.inf   # a non-finite guess (cte_1) stops that problem only
        r = m.solve_batch(st, cf, x_init=xb)
        assert r["status"][3] == -13 and r["iters"][3] == 0
        assert (np.delete(r["status"], 3) == 0).all()
