"""Adjoint sensitivities of solutions (b200mpc_solve_batch_vjp, not reference behaviour).  CPU tests run the host build
of the solver core (tests/hostsim/hostsim_sens.cpp) against a dense KKT solve built from the C port's evaluator and
against finite differences of the host-build solve; -m gpu runs the library's kernel against the host build and
checks the C ABI, the Python API and the autograd wrapper."""
import ctypes
import os

import numpy as np
import pytest

from conftest import golden, has_gpu

dp = ctypes.POINTER(ctypes.c_double)
PNAMES = ("ref_v", "w_cte", "w_epsi", "w_v", "w_delta", "w_a", "w_ddelta", "w_da")


def _p(a):
    return None if a is None else a.ctypes.data_as(dp)


def _coeffs(g):
    return g["coeffs"] if "coeffs" in g.files else g["fit"]


@pytest.fixture(scope="module")
def sens(_build_everything):
    """solve(state6, coeffs): the host-build solve with its multipliers (hostsim_solve_guess from the default start);
    vjp(...): hostsim_vjp, one problem."""
    import oracle_bindings as ob
    hs = os.path.join(ob.ROOT, "tests", "hostsim")
    lg = ctypes.CDLL(os.path.join(hs, "libhostsim_guess.so"))
    ls = ctypes.CDLL(os.path.join(hs, "libhostsim_sens.so"))
    ls.hostsim_vjp.argtypes = [ctypes.c_void_p, dp, dp, ctypes.c_int, dp, dp, dp, dp, ctypes.c_double, dp, dp, dp]

    class S:
        @staticmethod
        def solve(state6, coeffs, **params):
            p = ob.default_params(**params)
            N = p.N
            st = np.ascontiguousarray(state6, dtype=np.float64); c = np.ascontiguousarray(coeffs, dtype=np.float64)
            x = np.zeros(8 * N - 2); o8 = np.zeros(8); obj = ctypes.c_double(); it = ctypes.c_int(); m = np.zeros(10 * N - 4)
            rc = lg.hostsim_solve_guess(ctypes.byref(p), _p(st), _p(c), len(c), None, None, ctypes.c_double(1e-4), _p(x),
                                        _p(o8), ctypes.byref(obj), ctypes.byref(it), _p(m), 0)
            return dict(status=rc, x=x, out8=o8, obj=obj.value, mult=m)

        @staticmethod
        def vjp(state6, coeffs, x, mult, g_out8=None, g_traj=None, g_obj=0.0, **params):
            p = ob.default_params(**params)
            a = [np.ascontiguousarray(v, dtype=np.float64) if v is not None else None
                 for v in (state6, coeffs, x, mult, g_out8, g_traj)]
            gs, gc, gp = np.zeros(6), np.zeros(len(a[1])), np.zeros(8)
            rc = ls.hostsim_vjp(ctypes.byref(p), _p(a[0]), _p(a[1]), len(a[1]), _p(a[2]), _p(a[3]), _p(a[4]), _p(a[5]),
                                float(g_obj), _p(gs), _p(gc), _p(gp))
            return dict(status=rc, grad_state6=gs, grad_coeffs=gc, grad_params=gp)
    return S


def gbar_of(g_out8, g_traj, N):
    """The incoming gradient on the 8N-2 variables: g_traj plus g_out8 scattered onto s_1, delta_0, a_0."""
    g = np.zeros(8 * N - 2) if g_traj is None else np.array(g_traj, dtype=np.float64)
    if g_out8 is not None:
        g[np.arange(6) * N + 1] += g_out8[:6]
        g[6 * N] += g_out8[6]
        g[6 * N + N - 1] += g_out8[7]
    return g


def dense_vjp(state6, coeffs, x, mult, gbar, g_obj=0.0, N=25, h=1e-6):
    """grad = -[y_x; y_lam]^T dF/dtheta with K y = [gbar; 0] from the C port's evaluator, dense; dF/dtheta by central
    differences of the residual map (h), plus g_obj times the envelope term df/dtheta + lambda^T dc/dtheta."""
    import oracle_bindings as ob
    p = ob.default_params(N=N)
    M, n, m = N - 1, 8 * N - 2, 6 * N
    lam, zl, zu = mult[:m], mult[m:m + 2 * M], mult[m + 2 * M:]

    def ev(cf, **kw):
        f, grad, g, J, H = ob.port_eval(x, lam, cf, params=ob.default_params(N=N, **kw))
        return f, np.concatenate([grad + J.T @ lam, g]), g, J, H

    _, _, _, J, H = ev(coeffs)
    W = np.tril(H) + np.tril(H, -1).T   # port_eval returns the lower triangle
    b = np.repeat([p.delta_max, p.a_max], M)
    rel = 1e-8 * np.maximum(1.0, b)
    u = x[6 * N:]
    W[6 * N:, 6 * N:] += np.diag(zl / (u + b + rel) + zu / (b + rel - u))
    K = np.block([[W, J.T], [J, np.zeros((m, m))]])
    y = np.linalg.solve(K, np.concatenate([gbar, np.zeros(m)]))
    rows0 = np.arange(6) * N
    gs6 = y[n + rows0] - g_obj * lam[rows0]
    gc = np.zeros(len(coeffs))
    for i in range(len(coeffs)):
        def cd(hh):   # F is strongly nonlinear in the coefficients (x^3 with |x| up to ~100): Richardson below
            cp, cm = np.array(coeffs, dtype=np.float64), np.array(coeffs, dtype=np.float64)
            cp[i] += hh; cm[i] -= hh
            (_, Fp, gp, _, _), (_, Fm, gm, _, _) = ev(cp), ev(cm)
            return -y @ (Fp - Fm) / (2 * hh) + g_obj * lam @ (gp - gm) / (2 * hh)
        gc[i] = (4.0 * cd(h / 2) - cd(h)) / 3.0
    gpar = np.zeros(8)
    for i, name in enumerate(PNAMES):
        v = getattr(p, name)
        (fp, Fp, _, _, _), (fm, Fm, _, _, _) = ev(coeffs, **{name: v + h}), ev(coeffs, **{name: v - h})
        gpar[i] = -y @ (Fp - Fm) / (2 * h) + g_obj * (fp - fm) / (2 * h)
    return dict(grad_state6=gs6, grad_coeffs=gc, grad_params=gpar)


def _problems(n_each=16):
    out = []
    for name in ("roadmap_256.npz", "line_256.npz"):
        g = golden(name)
        for b in range(0, 256, 256 // n_each):
            out.append((g["states"][b], _coeffs(g)[b]))
    return out


def _rel(a, b):
    return float(np.abs(a - b).max() / max(1.0, np.abs(b).max()))


# ------------------------------------------------------------------------------------------------ CPU (host build)
def test_host_vjp_matches_the_dense_kkt_solve(sens):
    """32 problems, random incoming gradients on out8, traj and obj.  Both solve the same system; observed maxima,
    relative to max(1, |grad|): state6 3.4e-15, coefficients 1.9e-10, parameters 2.2e-9 (the last two: rounding of the
    dense reference's central differences of dF/dtheta)."""
    rng = np.random.default_rng(7)
    worst = 0.0
    for st, cf in _problems():
        r = sens.solve(st, cf)
        assert r["status"] == 0
        go8, gt, gob = rng.standard_normal(8), rng.standard_normal(198), float(rng.standard_normal())
        v = sens.vjp(st, cf, r["x"], r["mult"], go8, gt, gob)
        assert v["status"] == 0
        d = dense_vjp(st, cf, r["x"], r["mult"], gbar_of(go8, gt, 25), gob)
        for k in ("grad_state6", "grad_coeffs", "grad_params"):
            worst = max(worst, _rel(v[k], d[k]))
    print(f"host build vs dense KKT solve: max relative difference {worst:.2e}")
    assert worst < 1e-7, worst


def test_dense_reference_matches_finite_differences_of_the_solve(sens):
    """The dense reference (and so the VJP) is the derivative of the solver's output: central differences of the
    host-build solve at h = 1e-5 (default tol) within 1e-3 relative, and d obj / d state6 = -lambda at the rows of t = 0."""
    rng = np.random.default_rng(3)
    g = golden("roadmap_256.npz")
    for b in (0, 5, 17, 40, 99):
        st, cf = g["states"][b], g["fit"][b]
        r = sens.solve(st, cf)
        gt = rng.standard_normal(198)
        v = sens.vjp(st, cf, r["x"], r["mult"], None, gt, 0.0)
        d = dense_vjp(st, cf, r["x"], r["mult"], gt)
        assert _rel(v["grad_state6"], d["grad_state6"]) < 1e-6 and _rel(v["grad_coeffs"], d["grad_coeffs"]) < 1e-6
        h = 1e-5
        fd_s, fd_c, fd_obj = np.zeros(6), np.zeros(4), np.zeros(6)
        for k in range(6):
            sp, sm = st.copy(), st.copy()
            sp[k] += h; sm[k] -= h
            rp, rm = sens.solve(sp, cf), sens.solve(sm, cf)
            fd_s[k] = gt @ (rp["x"] - rm["x"]) / (2 * h)
            fd_obj[k] = (rp["obj"] - rm["obj"]) / (2 * h)
        for i in range(4):
            cp, cm = cf.copy(), cf.copy()
            cp[i] += h; cm[i] -= h
            fd_c[i] = gt @ (sens.solve(st, cp)["x"] - sens.solve(st, cm)["x"]) / (2 * h)
        assert _rel(d["grad_state6"], fd_s) < 1e-3, (b, d["grad_state6"], fd_s)
        assert _rel(d["grad_coeffs"], fd_c) < 1e-3, (b, d["grad_coeffs"], fd_c)
        env = sens.vjp(st, cf, r["x"], r["mult"], None, None, 1.0)["grad_state6"]
        np.testing.assert_allclose(env, -r["mult"][np.arange(6) * 25], rtol=0, atol=1e-12)
        assert _rel(env, fd_obj) < 1e-5, (b, env, fd_obj)


def test_parameter_gradients_match_finite_differences_of_the_solve(sens):
    """grad_params against central differences of the host-build solve with perturbed weights / ref_v."""
    import oracle_bindings as ob
    rng = np.random.default_rng(11)
    g = golden("roadmap_256.npz")
    st, cf = g["states"][5], g["fit"][5]
    r = sens.solve(st, cf)
    gt = rng.standard_normal(198)
    v = sens.vjp(st, cf, r["x"], r["mult"], None, gt, 0.5)
    p = ob.default_params()
    fd = np.zeros(8)
    for i, name in enumerate(PNAMES):
        h = 1e-5 * max(1.0, abs(getattr(p, name)))
        rp = sens.solve(st, cf, **{name: getattr(p, name) + h})
        rm = sens.solve(st, cf, **{name: getattr(p, name) - h})
        fd[i] = (gt @ (rp["x"] - rm["x"]) + 0.5 * (rp["obj"] - rm["obj"])) / (2 * h)
    assert _rel(v["grad_params"], fd) < 1e-3, (v["grad_params"], fd)


def test_failure_statuses(sens):
    g = golden("line_256.npz")
    st, cf = g["states"][0], g["coeffs"][0]
    r = sens.solve(st, cf)
    gt = np.ones(198)
    bad = gt.copy()
    bad[7] = np.nan
    v = sens.vjp(st, cf, r["x"], r["mult"], None, bad, 0.0)
    assert v["status"] == -13 and np.isnan(v["grad_state6"]).all() and np.isnan(v["grad_params"]).all()
    v = sens.vjp(st, cf, r["x"], r["mult"], None, gt, np.inf)
    assert v["status"] == -13 and np.isnan(v["grad_coeffs"]).all()
    # a negative bound multiplier: the control block of the adjoint factor is indefinite there
    m = r["mult"].copy()
    m[150 + 3] = -1e9
    v = sens.vjp(st, cf, r["x"], m, None, gt, 0.0)
    assert v["status"] == -3 and np.isnan(v["grad_state6"]).all()


def test_package_import_stays_torch_free():
    import subprocess
    import sys
    code = "import sys, udacitympc_b200; assert 'torch' not in sys.modules"
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.run([sys.executable, "-c", code], cwd=root, check=True)


# ------------------------------------------------------------------------------------------------ GPU
gpu = pytest.mark.skipif(not has_gpu(), reason="needs a CUDA device")


def _solve(mpc, st, cf):
    r = mpc.solve_batch(st, cf, want_traj=True, want_mult=True)
    return r


def _rand_grads(rng, B, nv):
    return rng.standard_normal((B, 8)), rng.standard_normal((B, nv)), rng.standard_normal(B)


@pytest.mark.gpu
@gpu
@pytest.mark.parametrize("name,N", [("roadmap_256.npz", 25), ("roadmap_N10_64.npz", 10), ("roadmap_N50_64.npz", 50),
                                    ("roadmap_N100_64.npz", 100)])
def test_device_vjp_matches_the_host_build(sens, name, N):
    """Observed maximum: about 1e-12 relative (FMA contraction differs between nvcc and g++)."""
    import udacitympc_b200 as mp
    g = golden(name)
    st, cf = g["states"], _coeffs(g)
    rng = np.random.default_rng(N)
    with mp.MPC(N=N) as mpc:
        r = _solve(mpc, st, cf)
        go8, gt, gob = _rand_grads(rng, len(st), mpc.num_vars)
        v = mpc.solve_batch_vjp(st, cf, r["traj"], r["mult"], go8, gt, gob, want_params=True)
    worst, n = 0.0, 0
    for b in range(len(st)):
        if r["status"][b] not in (0, 1):
            continue
        h = sens.vjp(st[b], cf[b], r["traj"][b], r["mult"][b], go8[b], gt[b], gob[b], N=N)
        assert v["status"][b] == h["status"] == 0, b
        for k in ("grad_state6", "grad_coeffs", "grad_params"):
            worst = max(worst, _rel(v[k][b], h[k]))
        n += 1
    assert n >= len(st) // 2
    print(f"device vs host build, {name}: max relative difference {worst:.2e} over {n} problems")
    assert worst < 1e-8, worst


@pytest.mark.gpu
@gpu
def test_host_and_device_entries_agree_bitwise_and_launch_once():
    import torch
    import udacitympc_b200 as mp
    g = golden("roadmap_256.npz")
    st, cf = g["states"], g["fit"]
    rng = np.random.default_rng(1)
    with mp.MPC() as mpc:
        r = _solve(mpc, st, cf)
        go8, gt, gob = _rand_grads(rng, 256, mpc.num_vars)
        v = mpc.solve_batch_vjp(st, cf, r["traj"], r["mult"], go8, gt, gob, want_params=True)
        d = lambda a: torch.as_tensor(np.ascontiguousarray(np.asarray(a, dtype=np.float64).T), device="cuda")
        ins = [d(st), d(cf), d(r["traj"]), d(r["mult"]), d(go8), d(gt), torch.as_tensor(gob, device="cuda")]
        gs, gc, gp = (torch.empty(k, 256, dtype=torch.float64, device="cuda") for k in (6, 4, 8))
        vs = torch.empty(256, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()   # the call below runs on the handle's own stream
        n0 = mpc.launch_count()
        mpc.solve_batch_vjp_device(256, ins[0].data_ptr(), ins[1].data_ptr(), 4, *[t.data_ptr() for t in ins[2:]],
                                   gs.data_ptr(), gc.data_ptr(), gp.data_ptr(), vs.data_ptr())
        mpc.wait()
        assert mpc.launch_count() == n0 + 1
        np.testing.assert_array_equal(gs.cpu().numpy().T, v["grad_state6"])
        np.testing.assert_array_equal(gc.cpu().numpy().T, v["grad_coeffs"])
        np.testing.assert_array_equal(gp.cpu().numpy().T, v["grad_params"])
        np.testing.assert_array_equal(vs.cpu().numpy(), v["status"])


@pytest.mark.gpu
@gpu
def test_bench_workload_gets_finite_gradients(sens):
    """65 536 problems of the benchmark's workload: every converged problem gets finite gradients, and a 512-problem
    sample matches the host build."""
    import sys
    import udacitympc_b200 as mp
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench
    rng = np.random.default_rng(5)
    with mp.MPC() as mpc:
        st, cf = bench.make_workload("roadmap", 65536, mpc=mpc)
        r = _solve(mpc, st, cf)
        go8 = rng.standard_normal((65536, 8))
        v = mpc.solve_batch_vjp(st, cf, r["traj"], r["mult"], go8, None, None, want_params=True)
    conv = (r["status"] == 0) | (r["status"] == 1)
    assert conv.mean() > 0.99
    assert (v["status"][conv] == 0).all()
    for k in ("grad_state6", "grad_coeffs", "grad_params"):
        assert np.isfinite(v[k][conv]).all(), k
    worst = 0.0
    for b in rng.choice(np.flatnonzero(conv), 512, replace=False):
        h = sens.vjp(st[b], cf[b], r["traj"][b], r["mult"][b], go8[b], None, 0.0)
        for k in ("grad_state6", "grad_coeffs", "grad_params"):
            worst = max(worst, _rel(v[k][b], h[k]))
    print(f"bench workload: {conv.sum()} converged, sample of 512 vs host build: max relative difference {worst:.2e}")
    assert worst < 1e-8, worst


@pytest.mark.gpu
@gpu
@pytest.mark.parametrize("where", ["cuda", "cpu"])
@pytest.mark.parametrize("shared", [False, True])
def test_autograd_equals_the_direct_vjp(where, shared):
    import torch
    import udacitympc_b200 as mp
    from udacitympc_b200 import autograd
    g = golden("roadmap_256.npz")
    st_np, cf_np = g["states"][:128], (g["fit"][3] if shared else g["fit"][:128])
    rng = np.random.default_rng(2)
    with mp.MPC() as mpc:
        st = torch.tensor(st_np, device=where, requires_grad=True)
        cf = torch.tensor(cf_np, device=where, requires_grad=True)
        out8, traj, obj, status = autograd.solve(mpc, st, cf)
        w8, wt, wo = (torch.tensor(a, device=where) for a in _rand_grads(rng, 128, mpc.num_vars))
        loss = (out8 * w8).sum() + (traj * wt).sum() + (obj * wo).sum()
        gs, gc = torch.autograd.grad(loss, (st, cf))
        r = _solve(mpc, st_np, cf_np)
        np.testing.assert_array_equal(traj.detach().cpu().numpy(), r["traj"])
        v = mpc.solve_batch_vjp(st_np, cf_np, r["traj"], r["mult"], w8.cpu().numpy(), wt.cpu().numpy(), wo.cpu().numpy())
    assert (status.cpu().numpy() == 0).all()
    np.testing.assert_array_equal(gs.cpu().numpy(), v["grad_state6"])
    if shared:
        np.testing.assert_allclose(gc.cpu().numpy(), v["grad_coeffs"].sum(0), rtol=0,
                                   atol=1e-12 * np.abs(v["grad_coeffs"]).sum(0).max())
    else:
        np.testing.assert_array_equal(gc.cpu().numpy(), v["grad_coeffs"])


@pytest.mark.gpu
@gpu
def test_vjp_after_pipelined_solves_equals_a_plain_handle():
    """A VJP queued after pipelined solves on other streams waits for their tails: same result as on a fresh handle."""
    import torch
    import udacitympc_b200 as mp
    g = golden("roadmap_256.npz")
    st, cf = g["states"], g["fit"]
    rng = np.random.default_rng(9)
    with mp.MPC() as plain:
        r = _solve(plain, st, cf)
        go8 = rng.standard_normal((256, 8))
        want = plain.solve_batch_vjp(st, cf, r["traj"], r["mult"], go8)
    import bench
    with mp.MPC() as mpc:
        mpc.set_pipeline(4, 1024)
        B = 16384
        bs, bc = bench.make_workload("roadmap", B, mpc=mpc)
        d_st = torch.as_tensor(np.ascontiguousarray(bs.T), device="cuda")
        d_cf = torch.as_tensor(np.ascontiguousarray(bc.T), device="cuda")
        streams = [torch.cuda.Stream() for _ in range(3)]
        torch.cuda.synchronize()
        outs = []
        for s in streams:
            o = torch.empty(8, B, dtype=torch.float64, device="cuda")
            outs.append(o)
            mpc.solve_batch_device(B, d_st.data_ptr(), d_cf.data_ptr(), 4, o.data_ptr(), stream=s.cuda_stream)
        got = mpc.solve_batch_vjp(st, cf, r["traj"], r["mult"], go8)
        torch.cuda.synchronize()
    for k in ("grad_state6", "grad_coeffs", "status"):
        np.testing.assert_array_equal(got[k], want[k])


@pytest.mark.gpu
@gpu
def test_argument_errors():
    import udacitympc_b200 as mp
    g = golden("roadmap_256.npz")
    st, cf = g["states"][:8], g["fit"][:8]
    with mp.MPC() as mpc:
        r = _solve(mpc, st, cf)
        lib, h = mpc._lib, mpc.handle
        P = lambda a: a.ctypes.data_as(dp)
        gs = np.zeros((8, 6))
        go8 = np.ones((8, 8))
        args = [P(st), P(cf), 4, P(r["traj"]), P(r["mult"])]
        rc = lib.b200mpc_solve_batch_vjp(h, 8, *args, None, None, None, P(gs), None, None, None)
        assert rc != 0 and b"no incoming gradient" in lib.b200mpc_last_error()
        assert lib.b200mpc_solve_batch_vjp(None, 8, *args, P(go8), None, None, P(gs), None, None, None) != 0
        assert lib.b200mpc_solve_batch_vjp(h, 0, *args, P(go8), None, None, P(gs), None, None, None) != 0
        bad = [P(st), P(cf), 5, P(r["traj"]), P(r["mult"])]
        assert lib.b200mpc_solve_batch_vjp(h, 8, *bad, P(go8), None, None, P(gs), None, None, None) != 0
        assert lib.b200mpc_solve_batch_vjp_device(h, 8, 1, 1, 1, 1, 1, None, None, None, None, None, None, None, None) != 0
        with pytest.raises(mp.B200MPCError):
            mpc.solve_batch_vjp(st, cf, r["traj"], r["mult"])
