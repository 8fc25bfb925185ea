"""-m gpu: parity of the CUDA path, called through the C ABI (udacitympc_b200 -> libb200mpc.so), against
  * golden vectors produced by the reference itself (tests/golden/make_golden.py), and
  * the CPU oracle (oracle/) on the same seeded inputs,
with the tolerances BASELINE.json's north_star states:
  actuators delta/a 1e-5 absolute, objective 1e-6 relative, predicted trajectory 1e-5,
  global_kinematic_model rollouts 1e-12, polyfit coefficients 1e-10."""
import ctypes
import os

import numpy as np
import pytest

import oracle_bindings as ob
import udacitympc_b200 as mp
from udacitympc_b200 import api, synth
from conftest import golden

pytestmark = pytest.mark.gpu

TOL_ACT, TOL_TRAJ, TOL_OBJ, TOL_ROLL, TOL_FIT = 1e-5, 1e-5, 1e-6, 1e-12, 1e-10


@pytest.fixture(scope="module")
def mpc():
    m = mp.MPC(device=0)
    yield m
    m.close()


def compare(r, g, sel=None, tight=1e-8, same_iters=0.98):
    sel = np.arange(len(g["status"])) if sel is None else np.asarray(sel)
    assert (r["status"][sel] == g["status"][sel]).all()
    np.testing.assert_allclose(r["out8"][sel, 6:], g["out8"][sel, 6:], rtol=0, atol=TOL_ACT)
    np.testing.assert_allclose(r["out8"][sel], g["out8"][sel], rtol=0, atol=TOL_TRAJ)
    np.testing.assert_allclose(r["traj"][sel], g["x"][sel], rtol=0, atol=TOL_TRAJ)
    assert (np.abs(r["cost"][sel] - g["obj"][sel]) <= TOL_OBJ * np.abs(g["obj"][sel])).all()
    # the device iterates track Ipopt's: in practice far tighter than the stated tolerances
    np.testing.assert_allclose(r["traj"][sel], g["x"][sel], rtol=0, atol=tight)
    assert (r["iters"][sel] == g["iters"][sel]).mean() >= same_iters


def test_config1_closed_loop_solve_calls(mpc):
    """solution/main.cpp:51-76 with MPC::Solve called 50 times through the drop-in class."""
    g = golden("config1_closed_loop.npz")
    coeffs = mp.polyfit([-100.0, 100.0], [-1.0, -1.0], 1, mpc=mpc)                      # main.cpp:25
    np.testing.assert_allclose(coeffs, g["coeffs"], rtol=0, atol=TOL_FIT)
    x, y, psi, v = -1.0, 10.0, 0.0, 10.0
    cte = mp.polyeval(coeffs, x, mpc=mpc) - y                                           # main.cpp:34
    epsi = psi - np.arctan(coeffs[1])
    state = np.array([x, y, psi, v, cte, epsi])
    for k in range(50):
        out = mpc.Solve(state, coeffs)
        assert len(out) == 8 and mpc.last_status == 0
        np.testing.assert_allclose(out, g["out8"][k], rtol=0, atol=1e-7)
        assert abs(mpc.last_cost - g["cost"][k]) <= TOL_OBJ * abs(g["cost"][k])
        assert mpc.last_iters == g["iters"][k]
        state = np.array(out[:6])


def test_config1_closed_loop_on_device(mpc):
    g = golden("config1_closed_loop.npz")
    r = mpc.closed_loop(g["states"][0], g["coeffs"], 50)
    np.testing.assert_allclose(r["hist8"][:, 0, :], g["out8"], rtol=0, atol=1e-7)
    assert (np.abs(r["cost"][:, 0] - g["cost"]) <= TOL_OBJ * np.abs(g["cost"])).all()
    assert (r["iters"][:, 0] == g["iters"]).all()


def test_closed_loop_of_several_vehicles_vs_reference_loop(mpc):
    """solution/main.cpp:51-76 for 12 vehicles with their own degree-3 references, 8 steps, on the device
    (b200mpc_closed_loop_batch) against the same loop run on the CPU one MPC::Solve at a time (make_golden.py --loops);
    its first step is the reference's own result in roadmap_256.npz."""
    g = golden("roadmap_256.npz")
    loop = golden("roadmap_closed_loop_12x8.npz")
    sel = np.arange(0, 240, 20)
    assert np.array_equal(loop["index"], sel)
    st, cf = g["states"][sel], g["fit"][sel]
    r = mpc.closed_loop(st, cf, 8)
    np.testing.assert_allclose(r["hist8"][0], g["out8"][sel], rtol=0, atol=1e-7)
    for j in range(len(sel)):
        for k in range(8):
            assert loop["status"][k, j] == 0
            np.testing.assert_allclose(r["hist8"][k, j], loop["out8"][k, j], rtol=0, atol=1e-7)
            assert abs(r["cost"][k, j] - loop["obj"][k, j]) <= TOL_OBJ * abs(loop["obj"][k, j])
            assert r["iters"][k, j] == loop["iters"][k, j]


def test_warm_started_closed_loop(mpc):
    """Optional warm start (off by default): same closed-loop trajectory as the cold-started reference loop within the
    solver tolerance, with fewer iterations; on both execution paths."""
    g = golden("config1_closed_loop.npz")
    for fb in (1 << 30, 0):   # cooperative kernel / per-pass kernels + cooperative finisher
        with mp.MPC(device=0) as m:
            m.set_solver_mode(0, 0, fb)
            cold = m.closed_loop(np.repeat(g["states"][:1], 3, axis=0), g["coeffs"], 50)
            m.set_warm_start(True, 1e-4)
            warm = m.closed_loop(np.repeat(g["states"][:1], 3, axis=0), g["coeffs"], 50)
        np.testing.assert_allclose(cold["hist8"][:, 0, :], g["out8"], rtol=0, atol=1e-7)
        np.testing.assert_allclose(warm["hist8"][:, 0, :], g["out8"], rtol=0, atol=1e-6)
        np.testing.assert_array_equal(warm["hist8"][:, 0, :], warm["hist8"][:, 2, :])
        assert (cold["iters"][:, 0] == g["iters"]).all()
        assert warm["iters"][:, 0].sum() < 0.5 * cold["iters"][:, 0].sum()


@pytest.mark.parametrize("name", ["line_256.npz", "roadmap_256.npz"])
@pytest.mark.parametrize("path", ["coop", "perpass", "fused"])
def test_random_problems_vs_reference(name, path):
    """Every execution path of the solver: cooperative warp-per-problem kernel (default for small batches), per-pass
    thread-per-problem kernels (default for large batches; forced here with fused_below = 0) and the fused
    thread-per-problem kernel."""
    g = golden(name)
    cf = g["coeffs"] if "coeffs" in g.files else g["fit"]
    with mp.MPC(device=0) as m:
        if path == "perpass":
            m.set_solver_mode(0, 12, 0)    # 12 rounds only: about half of the problems finish in the cooperative finisher
        elif path == "fused":
            m.set_solver_mode(1, 0, -1)
        r = m.solve_batch(g["states"], cf, want_traj=True)
    compare(r, g)


@pytest.mark.parametrize("path", ["default", "perpass"])
@pytest.mark.parametrize("N", [10, 50, 100])
def test_other_horizons(N, path):
    g = golden(f"roadmap_N{N}_64.npz")
    with mp.MPC(N=N) as m:
        if path == "perpass":   # per-pass kernels with batch compaction, 2 sub-batches, then the cooperative finisher
            m.set_solver_mode(0, 14, 0)
            m.set_compaction(0.9, 2)
            m.set_batch_split(2)
        r = m.solve_batch(g["states"], g["coeffs"], want_traj=True)
    sel = np.where((g["status"] == 0) & (g["used_restoration"] == 0))[0]
    assert len(sel) >= 56
    compare(r, g, sel)
    # the problems where the reference used its restoration phase: the library's default (soft restoration phase, then its
    # own restoration step, b200mpc_set_restoration mode 2) solves every one of them; all but at most one (N = 100) end in
    # the reference's local minimum (DESIGN.md 3)
    rest = np.setdiff1d(np.arange(64), sel)
    assert (r["status"][rest] == 0).all()
    same = np.abs(r["cost"][rest] - g["obj"][rest]) <= 1e-6 * np.abs(g["obj"][rest])
    assert same.sum() >= len(rest) - 1


def test_other_parameters():
    g = golden("line_params_64.npz")
    N, dt, Lf, ref_v, dmax, amax = g["params"]
    with mp.MPC(N=int(N), dt=dt, Lf=Lf, ref_v=ref_v, delta_max=dmax, a_max=amax) as m:
        r = m.solve_batch(g["states"], g["coeffs"], want_traj=True)
    sel = np.where((g["status"] == 0) & (g["used_restoration"] == 0))[0]
    assert len(sel) >= 40
    compare(r, g, sel, same_iters=0.9)   # a hard set (many regularised / backtracked solves): termination knife-edges


def test_weights_and_scaling_vs_port(mpc):
    kw = dict(w_cte=3.0, w_epsi=0.5, w_v=0.2, w_delta=10.0, w_a=2.0, w_ddelta=50.0, w_da=4.0)
    g = golden("line_256.npz")
    with mp.MPC(**kw) as m:
        r = m.solve_batch(g["states"][:32], g["coeffs"][:32], want_traj=True)
    for b in range(0, 32, 4):
        o = ob.port_solve(g["states"][b], g["coeffs"][b], params=ob.default_params(**kw))
        assert r["status"][b] == o["status"] and r["iters"][b] == o["iters"]
        np.testing.assert_allclose(r["traj"][b], o["x"], rtol=0, atol=1e-8)
    with mp.MPC(ref_v=6.0) as m:   # small gradients: the least-square multiplier estimate is kept (<= 1000)
        st6 = g["states"][:8].copy()
        st6[:, 3] = 5.0 + 0.2 * np.arange(8)
        r = m.solve_batch(st6, g["coeffs"][:8], want_traj=True)
        for b in range(8):
            o = ob.port_solve(st6[b], g["coeffs"][b], params=ob.default_params(ref_v=6.0))
            assert r["status"][b] == o["status"] and r["iters"][b] == o["iters"]
            np.testing.assert_allclose(r["traj"][b], o["x"], rtol=0, atol=1e-8)
    st = np.array([[0.0, 70.0, 0.1, 12.0, -71.0, 0.1]])   # objective scaling branch (IpGradientScaling.cpp:99-116)
    r = mpc.solve_batch(st, np.array([[-1.0, 0.0]]), want_traj=True)
    o = ob.port_solve(st[0], [-1.0, 0.0])
    assert r["status"][0] == o["status"] and r["iters"][0] == o["iters"]
    np.testing.assert_allclose(r["traj"][0], o["x"], rtol=0, atol=1e-8)
    assert abs(r["cost"][0] - o["obj"]) <= TOL_OBJ * abs(o["obj"])


def test_polyfit_known_answer_and_fixtures(mpc):
    from test_oracle_golden import QUIZ_X, QUIZ_Y, QUIZ_EXPECT, sig6
    c = mp.polyfit(QUIZ_X, QUIZ_Y, 3, mpc=mpc)
    assert [sig6(mp.polyeval(c, float(x), mpc=mpc)) for x in range(21)] == QUIZ_EXPECT   # polyfit/solution/main.cpp:33-54
    g = golden("polyfit_shapes.npz")
    for key in [k for k in g.files if k.startswith("fit_")]:
        _, m, order = key.split("_")
        fit = mp.polyfit_batch(g[f"xs_{m}_{order}"], g[f"ys_{m}_{order}"], int(order), mpc=mpc)
        np.testing.assert_allclose(fit, g[key], rtol=0, atol=TOL_FIT * max(1.0, np.abs(g[key]).max()))
    r = golden("roadmap_256.npz")
    np.testing.assert_allclose(mp.polyfit_batch(r["xs"], r["ys"], 3, mpc=mpc), r["fit"], rtol=0, atol=TOL_FIT)
    with pytest.raises(AssertionError):
        mp.polyfit([0.0, 1.0], [0.0, 1.0], 2, mpc=mpc)   # helpers.h:26
    with pytest.raises(mp.B200MPCError):
        mp.polyfit_batch(np.zeros((4, 3)), np.zeros((4, 3)), 3, mpc=mpc)


def test_kinematic_known_answer_and_fixtures(mpc):
    from test_oracle_golden import sig6
    nxt = mp.global_kinematic([0, 0, np.deg2rad(45), 1], [np.deg2rad(5), 1], 0.3, mpc=mpc)
    assert [sig6(v) for v in nxt] == [0.212132, 0.212132, 0.798488, 1.3]   # global_kinematic_model/solution/main.cpp:30
    g = golden("kinematic_256.npz")
    one = mp.rollout_batch(g["states"], g["act"][:, :1, :], 0.3, 2.0, mpc=mpc)
    np.testing.assert_allclose(one[:, 0, :], g["one_step"], rtol=0, atol=TOL_ROLL)
    roll = mp.rollout_batch(g["states"], g["act"], 0.3, 2.0, mpc=mpc)
    np.testing.assert_allclose(roll, g["rollout"], rtol=0, atol=TOL_ROLL)


def test_edge_batches(mpc):
    g = golden("line_256.npz")
    r0 = mpc.solve_batch(np.zeros((0, 6)), np.zeros((0, 2)))
    assert r0["out8"].shape == (0, 8)
    for B in (1, 31, 33, 65):   # ragged warps / blocks
        r = mpc.solve_batch(g["states"][:B], g["coeffs"][:B], want_traj=True)
        np.testing.assert_allclose(r["traj"], g["x"][:B], rtol=0, atol=1e-8)
    with pytest.raises(mp.B200MPCError):
        mpc.solve_batch(g["states"][:2], np.zeros((2, 5)))   # degree 4 unsupported
    with pytest.raises(mp.B200MPCError):
        mpc.solve_batch(g["states"][:2], np.zeros((2, 1)))
    # a quadratic (ncoef = 3) reference against the oracle
    cf = np.array([[0.5, -0.1, 0.004]])
    st = np.array([[0.0, 1.0, 0.05, 15.0, -0.5, 0.05 - np.arctan(-0.1)]])
    r = mpc.solve_batch(st, cf, want_traj=True)
    o = ob.port_solve(st[0], cf[0])
    np.testing.assert_allclose(r["traj"][0], o["x"], rtol=0, atol=1e-8)


def _ref_solve_one(a):
    o = ob.ref_solve(a[0], a[1])
    return o["x"], o["obj"], o["status"], o["iters"]


def test_full_size_batch_properties(mpc):
    """BASELINE size (65 536 problems): size-independent properties + a sample against the oracle."""
    B = 65536
    xs, ys = synth.roadmap_windows(B)
    fit = mp.polyfit_batch(xs, ys, 3, mpc=mpc)
    st = synth.roadmap_problems(B, fit)
    r = mpc.solve_batch(st, fit, want_traj=True)
    assert (r["status"] == 0).mean() > 0.999
    ok = r["status"] == 0
    N = 25
    T = r["traj"]
    X, Y, PSI, V = T[:, 0:N], T[:, N:2 * N], T[:, 2 * N:3 * N], T[:, 3 * N:4 * N]
    DEL, ACC = T[:, 6 * N:7 * N - 1], T[:, 7 * N - 1:]
    # bounds honoured exactly (honor_original_bounds), initial state pinned
    assert np.abs(DEL).max() <= 0.436332 and np.abs(ACC).max() <= 1.0
    np.testing.assert_allclose(T[:, [0, N, 2 * N, 3 * N, 4 * N, 5 * N]], st, rtol=0, atol=1e-12)
    # dynamic feasibility: rolling the bicycle model (K5) with the solution's own actuators reproduces x,y,psi,v
    roll = mp.rollout_batch(st[:, :4], np.stack([DEL, ACC], axis=2), 0.05, 2.67, mpc=mpc)
    err = np.abs(np.stack([X[:, 1:], Y[:, 1:], PSI[:, 1:], V[:, 1:]], axis=2) - roll).max(axis=(1, 2))
    assert err[ok].max() < 2e-6   # 1e-8 bound relaxation on a (IpOrigIpoptNLP.cpp:369-372) accumulates over 24 steps
    # returned objective = cost recomputed from the trajectory (MPC.cpp:57-76)
    cost = (T[:, 4 * N:5 * N] ** 2).sum(1) + (T[:, 5 * N:6 * N] ** 2).sum(1) + ((V - 40.0) ** 2).sum(1) + (DEL ** 2).sum(1) + \
        (ACC ** 2).sum(1) + (np.diff(DEL, axis=1) ** 2).sum(1) + (np.diff(ACC, axis=1) ** 2).sum(1)
    assert (np.abs(cost - r["cost"])[ok] <= 1e-6 * np.abs(cost[ok])).all()
    # out8 is the t=1 slice of the trajectory (MPC.cpp:253-256)
    np.testing.assert_array_equal(r["out8"][:, 0], X[:, 1]); np.testing.assert_array_equal(r["out8"][:, 6], DEL[:, 0])
    # determinism / idempotence, and sharding invariance (two halves == whole)
    r2 = mpc.solve_batch(st, fit, want_traj=False)
    np.testing.assert_array_equal(r2["out8"], r["out8"])
    h = B // 2
    ra, rb = mpc.solve_batch(st[:h], fit[:h]), mpc.solve_batch(st[h:], fit[h:])
    # (the hand-over to the cooperative kernel adapts to the batch, and the two kernels sum in different orders: the few
    # problems that finish on the other side of it may differ in the last bit)
    np.testing.assert_allclose(np.concatenate([ra["out8"], rb["out8"]]), r["out8"], rtol=0, atol=1e-13)
    np.testing.assert_array_equal(np.concatenate([ra["iters"], rb["iters"]]), r["iters"])
    with mp.MPC(device=0) as m:   # with a fixed hand-over point the halves reproduce the whole bit for bit
        m.set_solver_mode(0, 18, -1)
        whole = m.solve_batch(st, fit)
        ra, rb = m.solve_batch(st[:h], fit[:h]), m.solve_batch(st[h:], fit[h:])
    np.testing.assert_array_equal(np.concatenate([ra["out8"], rb["out8"]]), whole["out8"])
    # a strided sample against the CPU oracle (the C port; 40 ms per solve)
    for b in range(0, B, B // 24):
        o = ob.port_solve(st[b], fit[b])
        assert o["status"] == r["status"][b]
        np.testing.assert_allclose(r["traj"][b], o["x"], rtol=0, atol=1e-8)
        assert abs(o["obj"] - r["cost"][b]) <= TOL_OBJ * abs(o["obj"])
    # and a larger strided sample against the reference's own Ipopt + MUMPS binaries (oracle/_ref), all host cores
    if ob.ref_available():
        import multiprocessing as mpr
        idx = list(range(7, B, B // 512))
        with mpr.get_context("fork").Pool(min(16, os.cpu_count() or 1)) as pool:
            res = pool.map(_ref_solve_one, [(st[b], fit[b]) for b in idx])
        for b, (x, obj, status, iters) in zip(idx, res):
            assert status == r["status"][b] == 0
            np.testing.assert_allclose(r["traj"][b, 6 * N:], x[6 * N:], rtol=0, atol=TOL_ACT)
            np.testing.assert_allclose(r["traj"][b], x, rtol=0, atol=TOL_TRAJ)
            assert abs(obj - r["cost"][b]) <= TOL_OBJ * abs(obj)
            np.testing.assert_allclose(r["traj"][b], x, rtol=0, atol=1e-8)
        assert np.mean([r["iters"][b] == it for b, (_, _, _, it) in zip(idx, res)]) >= 0.99


def test_device_pointer_entry_and_multi_handle(mpc):
    import torch
    g = golden("line_256.npz")
    B = 256
    dev = torch.device("cuda", 0)
    st = torch.from_numpy(np.ascontiguousarray(g["states"].T)).to(dev)
    cf = torch.from_numpy(np.ascontiguousarray(g["coeffs"].T)).to(dev)
    out8 = torch.zeros((8, B), dtype=torch.float64, device=dev)
    traj = torch.zeros((198, B), dtype=torch.float64, device=dev)
    obj = torch.zeros(B, dtype=torch.float64, device=dev)
    status = torch.full((B,), -7, dtype=torch.int32, device=dev)
    iters = torch.zeros(B, dtype=torch.int32, device=dev)
    s = torch.cuda.current_stream()
    mpc.solve_batch_device(B, st.data_ptr(), cf.data_ptr(), 2, out8.data_ptr(), traj.data_ptr(), obj.data_ptr(),
                           status.data_ptr(), iters.data_ptr(), s.cuda_stream)
    torch.cuda.synchronize()
    np.testing.assert_allclose(traj.T.cpu().numpy(), g["x"], rtol=0, atol=1e-8)
    np.testing.assert_allclose(out8.T.cpu().numpy(), g["out8"], rtol=0, atol=1e-8)
    assert (status.cpu().numpy() == 0).all()
    ms, n = mpc.kernel_time_ms(reset=True)
    assert n == 0   # timing events are opt-in (b200mpc_set_timing)
    mpc.set_timing(True)
    mpc.solve_batch_device(B, st.data_ptr(), cf.data_ptr(), 2, out8.data_ptr(), traj.data_ptr(), obj.data_ptr(),
                           status.data_ptr(), iters.data_ptr(), s.cuda_stream)
    torch.cuda.synchronize()
    ms, n = mpc.kernel_time_ms(reset=True)
    mpc.set_timing(False)
    assert n == 1 and ms > 0
    # sharded over two handles (here both on device 0; on a multi-GPU box one per device)
    with mp.MPC(device=0) as m2:
        r = api.solve_batch_multi([mpc, m2], g["states"], g["coeffs"], want_traj=True)
    np.testing.assert_allclose(r["traj"], g["x"], rtol=0, atol=1e-8)


def test_fp64_peak_is_plausible(mpc):
    tf = mpc.fp64_peak_tflops()
    assert 5.0 < tf < 80.0, tf


def test_sweep_arithmetic_reciprocals_and_quotients_within_one_ulp(mpc):
    """The sweeps divide without the IEEE slow path (drcp / ddiv in mpc_core.cuh: rcp.approx.ftz.f64 + Newton steps).
    Against numpy's correctly rounded results: within 1 ulp for operands in the normal range (magnitudes 1e-150 ..
    1e150, the solver's slacks / determinants / step components live in 1e-25 .. 1e12), and the IEEE special values for a
    zero / infinite divisor (what the fraction-to-the-boundary rule relies on: such a candidate is never the minimum)."""
    rng = np.random.default_rng(7)
    n = 1 << 18
    sign = lambda k: np.where(rng.random(k) < 0.5, -1.0, 1.0)
    a = sign(n) * 10.0 ** rng.uniform(-150, 150, n)
    b = sign(n) * 10.0 ** rng.uniform(-150, 150, n)
    a[: n // 4] = sign(n // 4) * rng.uniform(0.0, 2.0, n // 4)          # the tau of the step-size rule, slack-sized operands
    b[: n // 4] = sign(n // 4) * 10.0 ** rng.uniform(-25, 12, n // 4)
    q, r = mpc.selftest_division(a, b)
    with np.errstate(over="ignore", under="ignore"):
        q_ref, r_ref = a / b, 1.0 / b
    ok = np.isfinite(q_ref) & (np.abs(q_ref) > 1e-290) & (np.abs(q_ref) < 1e290)
    assert ok.mean() > 0.8
    assert (np.abs(q[ok] - q_ref[ok]) <= np.spacing(np.abs(q_ref[ok]))).all()
    assert (np.abs(r - r_ref) <= np.spacing(np.abs(r_ref))).all()
    # special divisors
    a2 = np.array([1.0, -2.0, 0.99, 0.0, 3.0, -3.0, 1.0])
    b2 = np.array([0.0, 0.0, -0.0, 0.0, np.inf, np.inf, -np.inf])
    q2, r2 = mpc.selftest_division(a2, b2)
    assert q2[0] == np.inf and q2[1] == -np.inf and q2[2] == -np.inf and np.isnan(q2[3])
    assert q2[4] == 0.0 and q2[5] == 0.0 and q2[6] == 0.0
    assert r2[0] == np.inf and r2[2] == -np.inf and r2[4] == 0.0 and r2[6] == 0.0


def test_cpp_drop_in_closed_loop(tmp_path):
    """examples/mpc_to_line_main.cpp = the reference's solution/main.cpp loop on the C++ drop-in class
    (include/b200mpc/MPC.h): compiled with g++ against libb200mpc.so, its printed trace must match the golden one."""
    import os
    import re
    import subprocess
    from conftest import ROOT
    exe = str(tmp_path / "mpc_to_line")
    libdir = os.path.join(ROOT, "udacitympc_b200", "lib")
    subprocess.run(["g++", "-std=c++11", "-O2", "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "examples", "mpc_to_line_main.cpp"),
                    "-L" + libdir, "-lb200mpc", "-Wl,-rpath," + libdir, "-o", exe], check=True)
    out = subprocess.run([exe, str(tmp_path / "trace.csv")], check=True, capture_output=True, text=True).stdout
    g = golden("config1_closed_loop.npz")
    costs = [float(v) for v in re.findall(r"^Cost (\S+)$", out, flags=re.M)]
    assert len(costs) == 50
    np.testing.assert_allclose(costs, g["cost"], rtol=1e-5)   # iostream prints 6 significant digits
    for name, col in (("x", 0), ("y", 1), ("psi", 2), ("v", 3), ("cte", 4), ("epsi", 5), ("delta", 6), ("a", 7)):
        vals = [float(v) for v in re.findall(rf"^{name} = (\S+)$", out, flags=re.M)]
        assert len(vals) == 50
        np.testing.assert_allclose(vals, g["out8"][:, col], rtol=1e-5, atol=2e-6)
    assert (tmp_path / "trace.csv").read_text().count("\n") == 51


def test_config3_4096_line_problems_vs_reference(mpc):
    """BASELINE configs[2]: 4096 randomized degree-1 problems, every one against the reference binaries' answer."""
    g = golden("config3_line_4096.npz")
    st, cf = synth.line_problems(4096)
    r = mpc.solve_batch(st, cf)
    assert (r["status"] == g["status"]).all() and (g["status"] == 0).all()
    np.testing.assert_allclose(r["out8"][:, 6:], g["out8"][:, 6:], rtol=0, atol=TOL_ACT)
    np.testing.assert_allclose(r["out8"], g["out8"], rtol=0, atol=TOL_TRAJ)
    assert (np.abs(r["cost"] - g["obj"]) <= TOL_OBJ * np.abs(g["obj"])).all()
    np.testing.assert_allclose(r["out8"], g["out8"], rtol=0, atol=1e-8)
    assert (r["iters"] == g["iters"]).mean() >= 0.995


def roadmap_reference_oracle(pose, cl):
    """numpy restatement of the roadmap front-end (nearest centre-line point, 6-point window, global -> vehicle frame)
    with the oracle's polyfit.  The reference only sketches this step (custom_MPC.cpp:177-212, not runnable), so the
    selection/transform part is pinned by this restatement only; the fit is the pinned polyfit oracle."""
    x, y, psi, v = pose
    i = int(np.argmin((x - cl[:, 0]) ** 2 + (y - cl[:, 1]) ** 2))
    i = min(i, len(cl) - 6)
    dx, dy = cl[i:i + 6, 0] - x, cl[i:i + 6, 1] - y
    c, s = np.cos(psi), np.sin(psi)
    lx, ly = c * dx + s * dy, c * dy - s * dx
    cf = ob.port_polyfit(lx, ly, 3)
    return np.array([0, 0, 0, v, cf[0], -np.arctan(cf[1])]), cf


def test_roadmap_front_end_and_pipeline(mpc):
    cl = synth.roadmap_centerline()
    rng = np.random.default_rng(11)
    B = 512
    k = rng.integers(0, len(cl) - 7, size=B)
    seg = cl[k + 1] - cl[k]
    heading = np.arctan2(seg[:, 1], seg[:, 0])
    t = rng.random(B)
    pos = cl[k] + t[:, None] * seg + rng.normal(scale=1.0, size=(B, 2))
    poses = np.column_stack([pos, heading + rng.normal(scale=0.1, size=B), 5 + 30 * rng.random(B)])
    st, cf = mp.roadmap_reference_batch(poses, cl, mpc=mpc)
    for b in range(0, B, 7):
        so, co = roadmap_reference_oracle(poses[b], cl)
        np.testing.assert_allclose(cf[b], co, rtol=0, atol=1e-9 * max(1.0, np.abs(co).max()))
        np.testing.assert_allclose(st[b], so, rtol=0, atol=1e-9)
    # the whole pipeline on the device: pose -> reference polynomial -> MPC solve
    r = mpc.solve_batch(st, cf, want_traj=True)
    assert (r["status"] == 0).mean() > 0.99
    for b in range(0, B, 64):
        o = ob.port_solve(st[b], cf[b])
        assert o["status"] == r["status"][b]
        np.testing.assert_allclose(r["traj"][b], o["x"], rtol=0, atol=1e-8)
    with pytest.raises(mp.B200MPCError):
        mp.roadmap_reference_batch(poses, cl[:4], mpc=mpc)


def test_roadmap_front_end_vs_reference_fixture(mpc):
    """tests/golden/frontend_256.npz (make_golden.py --frontend): the reference's roadmap.csv, the nearest-point rule of
    custom_MPC.cpp:177-185, and the REFERENCE's polyfit (helpers.h:24-44, compiled from where it lies) on the 6 waypoints
    from there in the vehicle frame.  The roadmap file goes through the library's own reader."""
    import os
    g = golden("frontend_256.npz")
    cl, slope = mp.read_roadmap_csv(os.path.join(os.path.dirname(mp.__file__), "data", "roadmap.csv"))
    np.testing.assert_array_equal(cl, g["centerline"])
    st, cf = mp.roadmap_reference_batch(g["poses"], cl, mpc=mpc)
    # polyfit tolerance of north_star (1e-10), relative to the size of the coefficients of a fit
    scale = np.maximum(1.0, np.abs(g["coeffs"]).max(axis=1, keepdims=True))
    assert (np.abs(cf - g["coeffs"]) <= TOL_FIT * scale).all(), np.abs(cf - g["coeffs"]).max()
    np.testing.assert_allclose(st, g["state6"], rtol=0, atol=TOL_FIT * 10)
    # and through the solver: same MPC answers from the fixture's inputs and from the library's front-end
    a = mpc.solve_batch(st[:32], cf[:32])
    b = mpc.solve_batch(g["state6"][:32], g["coeffs"][:32])
    ok = (a["status"] == 0) & (b["status"] == 0)
    assert ok.sum() >= 28
    np.testing.assert_allclose(a["out8"][ok], b["out8"][ok], rtol=0, atol=TOL_TRAJ)


def test_cost_weights_vs_reference_binaries(mpc):
    """b200mpc_params.w_* against goldens made by the reference's Ipopt + MUMPS binaries on the weighted problem
    (tests/golden/weights_64.npz, make_golden.py --weights; TNLP weights in oracle/ref_build/mpc_tnlp.cpp)."""
    g = golden("weights_64.npz")
    for name in ("a", "b"):
        w = g[f"w_{name}"]
        kw = dict(w_cte=w[0], w_epsi=w[1], w_v=w[2], w_delta=w[3], w_a=w[4], w_ddelta=w[5], w_da=w[6])
        with mp.MPC(**kw) as m:
            for kind in ("line", "road"):
                r = m.solve_batch(g[f"{kind}_states"], g[f"{kind}_coeffs"], want_traj=True)
                gg = {k: g[f"{kind}_{name}_{k}"] for k in ("status", "out8", "x", "obj", "iters")}
                compare(r, gg)


def test_reference_shaped_solve_reads_two_coefficients_like_fg_eval():
    """MPC.cpp:117-118 uses coeffs[0] and coeffs[1] whatever the vector's length; the full polynomial is an option."""
    state = np.array([0.0, 0.0, 0.0, 12.0, -0.7, 0.05])
    c4 = np.array([-0.7, -0.05, 0.02, 0.002])
    with mp.MPC() as m, mp.MPC(full_polynomial=True) as mf:
        a = m.Solve(state, c4)
        b = m.Solve(state, c4[:2])
        assert a == b
        c = mf.Solve(state, c4)
        assert np.abs(np.array(c) - np.array(a)).max() > 1e-8   # the curvature terms change the solution
        np.testing.assert_allclose(c, m.solve_batch(state[None], c4[None])["out8"][0], rtol=0, atol=1e-12)


def test_multi_entry_point_rejects_mismatched_or_repeated_handles(mpc):
    """b200mpc_solve_batch_multi: shards write rows of one result array, so every handle must share the horizon /
    parameters, and a handle may not appear twice (two host threads on one workspace)."""
    st, cf = synth.line_problems(256)
    with mp.MPC(device=0, N=10) as other_n, mp.MPC(device=0, ref_v=30.0) as other_p, mp.MPC(device=0) as same:
        for bad in ([mpc, other_n], [mpc, other_p], [mpc, mpc], [mpc, same, mpc]):
            with pytest.raises(mp.B200MPCError) as e:
                api.solve_batch_multi(bad, st, cf)
            assert "handle" in str(e.value)
        same.set_restoration(1)
        with pytest.raises(mp.B200MPCError):
            api.solve_batch_multi([mpc, same], st, cf)
        same.set_restoration(2)
        # ragged split over three handles on one device (85 + 85 + 86 problems), and more handles than problems
        with mp.MPC(device=0) as third:
            r = api.solve_batch_multi([mpc, same, third], st, cf, want_traj=True)
            one = mpc.solve_batch(st, cf, want_traj=True)
            np.testing.assert_array_equal(r["status"], one["status"])
            np.testing.assert_array_equal(r["iters"], one["iters"])
            np.testing.assert_allclose(r["traj"], one["traj"], rtol=0, atol=1e-9)
            r2 = api.solve_batch_multi([mpc, same, third], st[:2], cf[:2])
            np.testing.assert_allclose(r2["out8"], one["out8"][:2], rtol=0, atol=1e-9)


def test_solves_on_one_handle_from_two_streams_are_serialised(mpc):
    """One workspace per handle: a second device call on another stream waits (on the device) for the first."""
    import torch
    dev = torch.device("cuda", 0)
    B = 4096
    sts, cfs = synth.line_problems(2 * B)
    outs = []
    strs = [torch.cuda.Stream(device=dev) for _ in range(2)]
    for k in range(2):
        st = torch.from_numpy(np.ascontiguousarray(sts[k * B:(k + 1) * B].T)).to(dev)
        cf = torch.from_numpy(np.ascontiguousarray(cfs[k * B:(k + 1) * B].T)).to(dev)
        out8 = torch.zeros((8, B), dtype=torch.float64, device=dev)
        status = torch.full((B,), -7, dtype=torch.int32, device=dev)
        outs.append((st, cf, out8, status))
    torch.cuda.synchronize()
    for rep in range(3):
        for k in range(2):
            st, cf, out8, status = outs[k]
            mpc.solve_batch_device(B, st.data_ptr(), cf.data_ptr(), 2, out8.data_ptr(), 0, 0, status.data_ptr(), 0, strs[k].cuda_stream)
    torch.cuda.synchronize()
    for k in range(2):
        ref = mpc.solve_batch(sts[k * B:(k + 1) * B], cfs[k * B:(k + 1) * B])
        assert (outs[k][3].cpu().numpy() == 0).all()
        np.testing.assert_allclose(outs[k][2].T.cpu().numpy(), ref["out8"], rtol=0, atol=1e-9)


def test_multi_device_sharding_in_one_process():
    """b200mpc_solve_batch_multi with one handle per GPU (contiguous index ranges, one host thread per device)."""
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    g = golden("config3_line_4096.npz")
    st, cf = synth.line_problems(4096)
    ms = [mp.MPC(device=d) for d in range(min(n, 4))]
    try:
        for fb in (0, 1 << 30):   # per-pass + cooperative finisher, cooperative only
            for m in ms:
                m.set_solver_mode(0, 0, fb)
            r = api.solve_batch_multi(ms, st, cf)
            assert (r["status"] == 0).all()
            np.testing.assert_allclose(r["out8"], g["out8"], rtol=0, atol=1e-8)
    finally:
        for m in ms:
            m.close()


def test_ragged_batch_on_the_throughput_path(mpc):
    """A batch that is not a multiple of the warp / block size through the per-pass kernels + finisher."""
    g = golden("config3_line_4096.npz")
    st, cf = synth.line_problems(4096)
    B = 4001
    r = mpc.solve_batch(st[:B], cf[:B])
    assert (r["status"] == 0).all()
    np.testing.assert_allclose(r["out8"], g["out8"][:B], rtol=0, atol=1e-8)


def test_internal_batch_split_does_not_change_results():
    """b200mpc_set_batch_split: the sub-batches of one call run on internal streams; every split gives bit-identical
    results (ragged batch, several closed-loop steps, trajectory output)."""
    st, cf = synth.line_problems(4096)
    B = 3999
    ref = None
    with mp.MPC(device=0) as m:
        m.set_solver_mode(0, 12, 0)   # per-pass kernels + cooperative finisher also for the small parts
        with pytest.raises(mp.B200MPCError):
            m.set_batch_split(5)
        for parts in (1, 2, 3, 4):
            m.set_batch_split(parts)
            r = m.solve_batch(st[:B], cf[:B], want_traj=True)
            loop = m.closed_loop(st[:300], cf[0], 3)
            if ref is None:
                ref = (r, loop)
                assert (r["status"] == 0).all()
                continue
            for k in ("out8", "traj", "cost", "status", "iters"):
                np.testing.assert_array_equal(r[k], ref[0][k])
            np.testing.assert_array_equal(loop["hist8"], ref[1]["hist8"])


def test_batch_compaction_does_not_change_results():
    """b200mpc_set_compaction: unfinished problems are moved to consecutive workspace slots between rounds (two
    regions, ping-pong); any threshold gives bit-identical results (1.0 = move after every round, whatever state the
    problems are in), also combined with the internal batch split, over several closed-loop steps, and when the
    finisher is the thread-per-problem kernel."""
    st, cf = synth.line_problems(4096)
    B = 3999
    with mp.MPC(device=0) as m:
        m.set_solver_mode(0, 20, 0)
        m.set_batch_split(1)
        m.set_compaction(0.0)
        ref = m.solve_batch(st[:B], cf[:B], want_traj=True)
        ref_loop = m.closed_loop(st[:300], cf[0], 3)
        assert (ref["status"] == 0).all()
        with pytest.raises(mp.B200MPCError):
            m.set_compaction(1.5)
        for frac, first, parts in ((0.7, 4, 1), (1.0, 1, 1), (0.99, 2, 2), (0.5, 8, 3), (0.9, 12, 4), (0.3, 1, 1)):
            m.set_compaction(frac, first)
            m.set_batch_split(parts)
            r = m.solve_batch(st[:B], cf[:B], want_traj=True)
            for k in ("out8", "traj", "cost", "status", "iters"):
                np.testing.assert_array_equal(r[k], ref[k], err_msg=f"{frac} {first} {parts} {k}")
            loop = m.closed_loop(st[:300], cf[0], 3)
            np.testing.assert_array_equal(loop["hist8"], ref_loop["hist8"])
    os.environ["B200MPC_NO_COOP"] = "1"
    try:
        with mp.MPC(device=0) as m:
            m.set_solver_mode(0, 14, 0)
            m.set_compaction(0.0)
            ref = m.solve_batch(st[:B], cf[:B], want_traj=True)
            m.set_compaction(0.95, 3)
            r = m.solve_batch(st[:B], cf[:B], want_traj=True)
    finally:
        del os.environ["B200MPC_NO_COOP"]
    for k in ("out8", "traj", "cost", "status", "iters"):
        np.testing.assert_array_equal(r[k], ref[k])


def test_overlapped_solves_are_deterministic():
    """The same 65 536-problem batch (bench.py's input set 3, which contains a 60+ iteration straggler) solved 12 times
    on three overlapped solver handles / streams: every result is bit-identical to the first one."""
    import torch
    B, S, reps = 65536, 3, 12
    xs, ys = synth.roadmap_windows(B, synth.MT19937_64(synth.SEED + 3000))
    dev = torch.device("cuda", 0)
    mpcs = [mp.MPC(device=0) for _ in range(S)]
    try:
        for h in mpcs:
            h.set_batch_split(1)
        fit = mp.polyfit_batch(xs, ys, 3, mpc=mpcs[0])
        st = synth.roadmap_problems(B, fit, synth.MT19937_64(synth.SEED + 3001))
        st_d = torch.from_numpy(np.ascontiguousarray(st.T)).to(dev)
        cf_d = torch.from_numpy(np.ascontiguousarray(fit.T)).to(dev)
        streams = [torch.cuda.Stream(device=dev) for _ in range(S)]
        outs = [dict(out8=torch.empty((8, B), dtype=torch.float64, device=dev), status=torch.empty(B, dtype=torch.int32, device=dev),
                     iters=torch.empty(B, dtype=torch.int32, device=dev)) for _ in range(reps)]
        torch.cuda.synchronize()
        for i, o in enumerate(outs):
            mpcs[i % S].solve_batch_device(B, st_d.data_ptr(), cf_d.data_ptr(), 4, o["out8"].data_ptr(), 0, 0, o["status"].data_ptr(),
                                           o["iters"].data_ptr(), streams[i % S].cuda_stream)
        torch.cuda.synchronize()
        assert int((outs[0]["status"] != 0).sum()) == 0
        assert int(outs[0]["iters"].max()) >= 40   # the straggler is in the set
        for o in outs[1:]:
            assert torch.equal(o["out8"], outs[0]["out8"]) and torch.equal(o["iters"], outs[0]["iters"])
            assert torch.equal(o["status"], outs[0]["status"])
        # the straggler against its one-at-a-time CPU solve (make_golden.py --loops)
        j = int(outs[0]["iters"].argmax())
        r = golden("straggler_set3.npz")
        assert j == r["index"]
        np.testing.assert_allclose(st[j], r["state"], rtol=0, atol=1e-9)
        np.testing.assert_allclose(fit[j], r["coeffs"], rtol=0, atol=1e-9)
        got = outs[0]["out8"][:, j].cpu().numpy()
        print("straggler", j, "iters", int(outs[0]["iters"][j]), "CPU iters", r["iters"], "status", r["status"])
        assert r["status"] == 0
        np.testing.assert_allclose(got[6:], [r["x"][6 * 25], r["x"][7 * 25 - 1]], rtol=0, atol=TOL_ACT)
        np.testing.assert_allclose(got[:6], [r["x"][k * 25 + 1] for k in range(6)], rtol=0, atol=TOL_TRAJ)
    finally:
        for h in mpcs:
            h.close()


def test_asynchronous_host_buffer_calls_from_one_thread(mpc):
    """b200mpc_solve_batch_async + b200mpc_wait: one host thread keeps three handles busy from pinned buffers; results are
    those of the blocking call."""
    import torch
    B = 8192
    sts, cfs = synth.line_problems(3 * B)
    ref = [mpc.solve_batch(sts[k * B:(k + 1) * B], cfs[k * B:(k + 1) * B]) for k in range(3)]
    lib = mp.load_library()
    dp, ip = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int)
    hs = [mp.MPC(device=0) for _ in range(3)]
    try:
        bufs = []
        for k in range(3):
            bufs.append(dict(st=torch.from_numpy(np.ascontiguousarray(sts[k * B:(k + 1) * B])).pin_memory(),
                             cf=torch.from_numpy(np.ascontiguousarray(cfs[k * B:(k + 1) * B])).pin_memory(),
                             out8=torch.zeros((B, 8), dtype=torch.float64).pin_memory(), obj=torch.zeros(B, dtype=torch.float64).pin_memory(),
                             status=torch.full((B,), -7, dtype=torch.int32).pin_memory(), iters=torch.zeros(B, dtype=torch.int32).pin_memory()))
        for rep in range(2):
            for k, (h, b) in enumerate(zip(hs, bufs)):
                rc = lib.b200mpc_solve_batch_async(h.handle, B, ctypes.cast(b["st"].data_ptr(), dp), ctypes.cast(b["cf"].data_ptr(), dp), 2,
                                                   ctypes.cast(b["out8"].data_ptr(), dp), None, ctypes.cast(b["obj"].data_ptr(), dp),
                                                   ctypes.cast(b["status"].data_ptr(), ip), ctypes.cast(b["iters"].data_ptr(), ip))
                assert rc == 0, lib.b200mpc_last_error()
            for h in hs:
                h.wait()
        for k, b in enumerate(bufs):
            assert (b["status"].numpy() == 0).all()
            assert (b["iters"].numpy() == ref[k]["iters"]).all()
            np.testing.assert_allclose(b["out8"].numpy(), ref[k]["out8"], rtol=0, atol=1e-12)
            np.testing.assert_allclose(b["obj"].numpy(), ref[k]["cost"], rtol=1e-13, atol=0)
        assert lib.b200mpc_wait(None) == -1
    finally:
        for h in hs:
            h.close()


def test_pipelined_solves_on_one_handle_match_plain_solves():
    """b200mpc_set_pipeline: batches issued on different streams to ONE handle (bulk in the main workspace, the last
    unfinished problems in small tail contexts, overlapped with the next bulk) give the results of plain solves: same
    status and iteration counts, solution to 1e-9 (a hand-over between the thread sweeps and the cooperative kernel may
    change last bits).  Three different batches, N = 25 and N = 50, depth 3 < number of calls (contexts are reused)."""
    import torch
    dev = torch.device("cuda", 0)
    for N, B, slots in ((25, 16384, 1024), (50, 8192, 512), (25, 65536, 4096)):
        sets = []
        with mp.MPC(device=0, N=N) as plain:
            for k in range(3):
                xs, ys = synth.roadmap_windows(B, synth.MT19937_64(synth.SEED + 500 + k))
                fit = mp.polyfit_batch(xs, ys, 3, mpc=plain)
                st = synth.roadmap_problems(B, fit, synth.MT19937_64(synth.SEED + 600 + k))
                sets.append((st, fit, plain.solve_batch(st, fit)))
        with mp.MPC(device=0, N=N) as piped:
            piped.set_batch_split(1)
            piped.set_pipeline(3, slots)
            streams = [torch.cuda.Stream(device=dev) for _ in range(4)]
            d_in = [(torch.from_numpy(np.ascontiguousarray(st.T)).to(dev), torch.from_numpy(np.ascontiguousarray(cf.T)).to(dev)) for st, cf, _ in sets]
            calls = 8
            outs = [dict(out8=torch.zeros((8, B), dtype=torch.float64, device=dev), obj=torch.zeros(B, dtype=torch.float64, device=dev),
                         status=torch.full((B,), -7, dtype=torch.int32, device=dev), iters=torch.zeros(B, dtype=torch.int32, device=dev))
                    for _ in range(calls)]
            torch.cuda.synchronize()
            for i, o in enumerate(outs):
                st_d, cf_d = d_in[i % 3]
                piped.solve_batch_device(B, st_d.data_ptr(), cf_d.data_ptr(), 4, o["out8"].data_ptr(), 0, o["obj"].data_ptr(),
                                         o["status"].data_ptr(), o["iters"].data_ptr(), streams[i % 4].cuda_stream)
            torch.cuda.synchronize()
            for i, o in enumerate(outs):
                ref = sets[i % 3][2]
                assert (o["status"].cpu().numpy() == ref["status"]).all(), (N, i)
                assert (o["iters"].cpu().numpy() == ref["iters"]).mean() > 0.999, (N, i)
                np.testing.assert_allclose(o["out8"].T.cpu().numpy(), ref["out8"], rtol=0, atol=1e-9)
                np.testing.assert_allclose(o["obj"].cpu().numpy(), ref["cost"], rtol=1e-12, atol=0)
            # a plain host-buffer call on the same handle afterwards (smaller than the tail: not pipelined) still works
            small = piped.solve_batch(sets[0][0][:256], sets[0][1][:256])
            np.testing.assert_allclose(small["out8"], sets[0][2]["out8"][:256], rtol=0, atol=1e-9)


def test_invalid_numbers_are_reported_per_problem():
    """NaN / Inf inputs: status -13 (Ipopt's Invalid_Number_Detected) for those problems only, on both paths."""
    g = golden("line_256.npz")
    st, cf = g["states"][:64].copy(), g["coeffs"][:64].copy()
    st[3, 1] = np.nan
    st[17, 3] = np.inf
    cf[40, 0] = np.nan
    bad = np.array([3, 17, 40])
    good = np.setdiff1d(np.arange(64), bad)
    for fb in (1 << 30, 0):   # cooperative kernel / per-pass kernels
        with mp.MPC(device=0) as m:
            m.set_solver_mode(0, 0, fb)
            r = m.solve_batch(st, cf, want_traj=True)
        assert (r["status"][bad] == -13).all() and (r["iters"][bad] == 0).all()
        assert (r["status"][good] == g["status"][good]).all()
        np.testing.assert_allclose(r["traj"][good], g["x"][good], rtol=0, atol=1e-8)


def test_plain_launches_and_changing_batch_sizes():
    """B200MPC_NO_GRAPHS=1 (plain launches instead of CUDA-graph replay, including the fork / join of a split call) gives
    the same results; one handle serves changing batch sizes (its workspace grows, graphs are re-captured)."""
    st, cf = synth.line_problems(8192)
    with mp.MPC(device=0) as m:
        a = m.solve_batch(st[:4096], cf[:4096])
        b = m.solve_batch(st, cf)                      # larger batch: the workspace is reallocated
        c = m.solve_batch(st[:4096], cf[:4096])        # back to the first size
        d = m.solve_batch(st[:100], cf[:100])          # latency path on the same handle
    for k in ("out8", "cost", "status", "iters"):
        np.testing.assert_array_equal(a[k], c[k])
        np.testing.assert_array_equal(a[k][:100], d[k]) if k in ("status", "iters") else None
    np.testing.assert_allclose(b["out8"][:4096], a["out8"], rtol=0, atol=1e-9)
    np.testing.assert_allclose(d["out8"], a["out8"][:100], rtol=0, atol=1e-9)
    os.environ["B200MPC_NO_GRAPHS"] = "1"
    try:
        with mp.MPC(device=0) as m:
            e = m.solve_batch(st, cf)
    finally:
        del os.environ["B200MPC_NO_GRAPHS"]
    for k in ("out8", "cost", "status", "iters"):
        np.testing.assert_array_equal(e[k], b[k])


def test_long_horizon_falls_back_to_the_thread_finisher():
    """From N = 205 on the cooperative kernel does not fit its shared memory (N = 204 is the last horizon that does, with
    one problem per block): the fused thread-per-problem kernel finishes the batch.  No oracle is fast enough at this
    size; check the size-independent properties instead."""
    N = 205
    st, cf = synth.line_problems(40)
    with mp.MPC(device=0, N=N, max_iter=400) as m:
        r = m.solve_batch(st, cf, want_traj=True)
        m.set_solver_mode(0, 12, 0)
        r2 = m.solve_batch(st, cf, want_traj=True)
    assert np.isin(r["status"], [0, 1, -1, -2]).all() and (r["status"] == 0).sum() >= 20
    np.testing.assert_array_equal(r["status"], r2["status"])
    ok = r["status"] == 0
    np.testing.assert_allclose(r["traj"][ok], r2["traj"][ok], rtol=0, atol=1e-9)   # both launch sequences, same answer
    T = r["traj"][ok]
    DEL, ACC = T[:, 6 * N:7 * N - 1], T[:, 7 * N - 1:]
    assert np.abs(DEL).max() <= 0.436332 and np.abs(ACC).max() <= 1.0
    with mp.MPC(device=0) as m0:
        roll = mp.rollout_batch(st[ok][:, :4], np.stack([DEL, ACC], axis=2), 0.05, 2.67, mpc=m0)
    err = np.abs(np.stack([T[:, 1:N], T[:, N + 1:2 * N], T[:, 2 * N + 1:3 * N], T[:, 3 * N + 1:4 * N]], axis=2) - roll).max()
    assert err < 1e-4


def test_long_solves_keep_every_filter_entry():
    """Extreme initial states (|cte| up to 80 m, 40-130 iterations): the filter grows beyond 8 entries; it lives in its own
    workspace record (41 entries) and moves with the problem in the batch compaction.  Same solutions as the reference
    binaries (these solves are sensitive: the iteration count is required to agree on two thirds only)."""
    g = golden("long_filter_N25_12.npz")
    for reps in (1, 300):   # cooperative kernel alone / per-pass kernels with compaction, then the finisher
        st, cf = np.tile(g["states"], (reps, 1)), np.tile(g["coeffs"], (reps, 1))
        with mp.MPC() as m:
            if reps > 1:
                m.set_solver_mode(0, 30, 0)
                m.set_compaction(0.9, 2)
            r = m.solve_batch(st, cf, want_traj=True)
        assert (r["status"] == 0).all()
        same = (np.abs(r["traj"][:12] - g["x"]).max(axis=1) <= TOL_TRAJ) & (np.abs(r["cost"][:12] - g["obj"]) <= TOL_OBJ * np.abs(g["obj"]))
        assert same.sum() >= 10, same
        assert (r["iters"][:12] == g["iters"]).sum() >= 8
