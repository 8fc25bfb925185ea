"""-m "not gpu": the solver core that the CUDA kernel runs (udacitympc_b200/csrc/mpc_core.cuh), compiled for the
host by tests/hostsim, against the reference's golden vectors.  This is the algorithm check that can run in the
GPU-less build container; the same comparisons run on the device in test_gpu_parity.py."""
import numpy as np
import pytest

from conftest import golden

TOL_ACT = 1e-5    # north_star: actuators delta/a within 1e-5 absolute
TOL_TRAJ = 1e-5   # predicted trajectory within 1e-5
TOL_OBJ = 1e-6    # objective within 1e-6 relative


def check(r, g, b, tight=True):
    assert r["status"] == g["status"][b]
    np.testing.assert_allclose(r["out8"][6:], g["out8"][b][6:], rtol=0, atol=TOL_ACT)
    np.testing.assert_allclose(r["x"], g["x"][b], rtol=0, atol=TOL_TRAJ)
    assert abs(r["obj"] - g["obj"][b]) <= TOL_OBJ * abs(g["obj"][b])
    if tight:   # the iterates track Ipopt's, so in practice the agreement is ~1e-12
        np.testing.assert_allclose(r["x"], g["x"][b], rtol=0, atol=1e-8)
    return int(r["iters"] == g["iters"][b])


def usable(g, b):
    """The restoration phase is not implemented (SURVEY 2.2 #11): problems where the reference needed it, or
    did not converge, return status -2 here and are excluded from the parity comparison."""
    return g["status"][b] == 0 and not g["used_restoration"][b]


def test_config1_closed_loop(hostsim):
    g = golden("config1_closed_loop.npz")
    state = g["states"][0].copy()
    for k in range(50):
        r = hostsim.solve(state, g["coeffs"])
        assert r["status"] == 0 and r["iters"] == g["iters"][k]
        np.testing.assert_allclose(r["out8"], g["out8"][k], rtol=0, atol=1e-8)
        assert abs(r["obj"] - g["cost"][k]) <= TOL_OBJ * abs(g["cost"][k])
        state = r["out8"][:6].copy()   # main.cpp:66


@pytest.mark.parametrize("name", ["line_256.npz", "roadmap_256.npz"])
def test_random_problems(hostsim, name):
    g = golden(name)
    cf = g["coeffs"] if "coeffs" in g.files else g["fit"]
    same = sum(check(hostsim.solve(g["states"][b], cf[b]), g, b) for b in range(256))
    assert same >= 254   # identical interior-point iteration counts (a knife-edge termination test may flip one)


@pytest.mark.parametrize("N", [10, 50, 100])
def test_other_horizons(hostsim, N):
    g = golden(f"roadmap_N{N}_64.npz")
    n_cmp = 0
    for b in range(64):
        if not usable(g, b):
            continue
        check(hostsim.solve(g["states"][b], g["coeffs"][b], N=N), g, b)
        n_cmp += 1
    assert n_cmp >= 56


def test_other_parameters(hostsim):
    g = golden("line_params_64.npz")
    N, dt, Lf, ref_v, dmax, amax = g["params"]
    n_cmp = same = 0
    for b in range(64):
        r = hostsim.solve(g["states"][b], g["coeffs"][b], N=int(N), dt=dt, Lf=Lf, ref_v=ref_v, delta_max=dmax, a_max=amax)
        if not usable(g, b):
            assert r["status"] in (0, -2)
            continue
        same += check(r, g, b)
        n_cmp += 1
    assert n_cmp >= 40 and same >= n_cmp - 2


def test_rare_paths_match_oracle(hostsim):
    """Inertia correction, backtracking and second-order correction are rare at N=25; N=50 problems from the
    golden set that used them (but not restoration) must still track the reference."""
    g = golden("roadmap_N50_64.npz")
    sel = [b for b in range(64) if g["status"][b] == 0 and not g["used_restoration"][b] and (g["max_regu"][b] > 0 or g["max_ls_trials"][b] > 1)]
    for b in sel:
        check(hostsim.solve(g["states"][b], g["coeffs"][b], N=50), g, b)


def test_objective_scaling_branch(hostsim):
    """|cte0| > 50 switches Ipopt's gradient-based objective scaling on (IpGradientScaling.cpp:99-116)."""
    import oracle_bindings as ob
    st = [0.0, 70.0, 0.1, 12.0, -71.0, 0.1]
    r = hostsim.solve(st, [-1.0, 0.0])
    o = ob.port_solve(st, [-1.0, 0.0])
    assert r["status"] == o["status"] and r["iters"] == o["iters"]
    np.testing.assert_allclose(r["x"], o["x"], rtol=0, atol=1e-8)
    assert abs(r["obj"] - o["obj"]) <= 1e-9 * abs(o["obj"])


def test_weights_against_port(hostsim):
    """Non-unit cost weights (not expressible through the reference TNLP driver) against the C port."""
    import oracle_bindings as ob
    kw = dict(w_cte=3.0, w_epsi=0.5, w_v=0.2, w_delta=10.0, w_a=2.0, w_ddelta=50.0, w_da=4.0)
    g = golden("line_256.npz")
    for b in range(0, 64, 8):
        r = hostsim.solve(g["states"][b], g["coeffs"][b], **kw)
        o = ob.port_solve(g["states"][b], g["coeffs"][b], params=ob.default_params(**kw))
        assert r["status"] == o["status"] and r["iters"] == o["iters"]
        np.testing.assert_allclose(r["x"], o["x"], rtol=0, atol=1e-8)


def test_per_pass_state_persistence(hostsim):
    """mode 1 = every pass on a fresh Solver whose scalars come from the workspace record (what the per-pass CUDA
    kernels do): must give bit-identical results to the single-object loop (mode 0), including on problems that
    take the rare paths (regularisation, backtracking, second-order correction)."""
    sets = [("line_256.npz", {}, range(0, 256, 4)), ("roadmap_N50_64.npz", dict(N=50), range(64))]
    g = golden("line_params_64.npz")
    N, dt, Lf, ref_v, dmax, amax = g["params"]
    sets.append(("line_params_64.npz", dict(N=int(N), dt=dt, Lf=Lf, ref_v=ref_v, delta_max=dmax, a_max=amax), range(64)))
    for name, kw, idx in sets:
        g = golden(name)
        cf = g["coeffs"] if "coeffs" in g.files else g["fit"]
        for b in idx:
            a = hostsim.solve(g["states"][b], cf[b], mode=0, **kw)
            c = hostsim.solve(g["states"][b], cf[b], mode=1, **kw)
            assert a["status"] == c["status"] and a["iters"] == c["iters"]
            np.testing.assert_array_equal(a["x"], c["x"])
            assert a["obj"] == c["obj"]


def test_batch_compaction_moves_everything_a_problem_owns(hostsim):
    """mode -1 / -2: as mode 1, with the problem moved to a NaN-poisoned workspace by repack_problem (the batch
    compaction of the per-pass path) after every round / after every pass, i.e. in every state a problem can be in:
    bit-identical results, including the rare paths (regularisation, backtracking, second-order correction) and the
    kept least-square multiplier estimate."""
    sets = [("line_256.npz", {}, range(0, 256, 8)), ("roadmap_256.npz", {}, range(0, 256, 8)), ("roadmap_N50_64.npz", dict(N=50), range(64))]
    g = golden("line_params_64.npz")
    N, dt, Lf, ref_v, dmax, amax = g["params"]
    sets.append(("line_params_64.npz", dict(N=int(N), dt=dt, Lf=Lf, ref_v=ref_v, delta_max=dmax, a_max=amax), range(64)))
    sets.append(("line_256.npz", dict(ref_v=6.0), range(0, 6)))
    for name, kw, idx in sets:
        g = golden(name)
        cf = g["coeffs"] if "coeffs" in g.files else g["fit"]
        for b in idx:
            a = hostsim.solve(g["states"][b], cf[b], mode=0, **kw)
            for mode in (-1, -2):
                c = hostsim.solve(g["states"][b], cf[b], mode=mode, **kw)
                assert a["status"] == c["status"] and a["iters"] == c["iters"], (name, b, mode)
                np.testing.assert_array_equal(a["x"], c["x"])
                assert a["obj"] == c["obj"]


def test_least_square_multiplier_estimate_is_kept_when_small(hostsim):
    """With a small reference speed the least-square multiplier estimate stays below constr_mult_init_max = 1000 and
    Ipopt keeps it (IpDefaultIterateInitializer.cpp:651-718); with the reference's ref_v = 40 it is discarded."""
    import oracle_bindings as ob
    g = golden("line_256.npz")
    for b in range(6):
        st = g["states"][b].copy()
        st[3] = 5.0 + 0.2 * b
        for mode in (0, 1, 2, 4, 5, 6):
            r = hostsim.solve(st, g["coeffs"][b], mode=mode, ref_v=6.0)
            o = ob.port_solve(st, g["coeffs"][b], params=ob.default_params(ref_v=6.0))
            assert r["status"] == o["status"] and r["iters"] == o["iters"]
            np.testing.assert_allclose(r["x"], o["x"], rtol=0, atol=1e-8)


def test_config3_sample(hostsim):
    from udacitympc_b200 import synth
    g = golden("config3_line_4096.npz")
    st, cf = synth.line_problems(4096)
    for b in range(0, 4096, 16):
        r = hostsim.solve(st[b], cf[b])
        assert r["status"] == g["status"][b] and r["iters"] == g["iters"][b]
        np.testing.assert_allclose(r["out8"], g["out8"][b], rtol=0, atol=1e-8)
        assert abs(r["obj"] - g["obj"][b]) <= TOL_OBJ * abs(g["obj"][b])


def test_cooperative_solver_matches_thread_version(hostsim):
    """The warp-per-problem (latency path) solver, emulated lane by lane on the host: from the start (mode 2) and
    taking a problem over from the thread version after k sweeps (mode 3+k), in whatever phase it is in."""
    sets = [("line_256.npz", {}, range(0, 256, 8)), ("roadmap_256.npz", {}, range(0, 256, 8)), ("roadmap_N50_64.npz", dict(N=50), range(0, 64, 2))]
    g = golden("line_params_64.npz")
    N, dt, Lf, ref_v, dmax, amax = g["params"]
    sets.append(("line_params_64.npz", dict(N=int(N), dt=dt, Lf=Lf, ref_v=ref_v, delta_max=dmax, a_max=amax), range(0, 64, 2)))
    for name, kw, idx in sets:
        g = golden(name)
        cf = g["coeffs"] if "coeffs" in g.files else g["fit"]
        for b in idx:
            a = hostsim.solve(g["states"][b], cf[b], mode=0, **kw)
            for mode in (2, 4, 5, 6, 3 + 3 * 7, 3 + 3 * 11 + 1, 3 + 3 * 30 + 2):
                c = hostsim.solve(g["states"][b], cf[b], mode=mode, **kw)
                assert a["status"] == c["status"] and a["iters"] == c["iters"], (name, b, mode)
                np.testing.assert_allclose(a["x"], c["x"], rtol=0, atol=1e-10)
                assert abs(a["obj"] - c["obj"]) <= 1e-12 * abs(a["obj"])


def test_warm_started_closed_loop_reaches_the_same_trajectory(hostsim):
    """Warm start (off by default; not reference behaviour): the 50-step closed loop of config 1 follows the cold-start
    (= reference) trajectory within the solver tolerance with far fewer interior-point iterations."""
    import ctypes
    import oracle_bindings as ob
    g = golden("config1_closed_loop.npz")
    dp, ip = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int)

    def loop(warm, mu):
        p = ob.default_params()
        st = np.ascontiguousarray(g["states"][0]); c = np.ascontiguousarray(g["coeffs"])
        h = np.zeros((50, 8)); it = np.zeros(50, dtype=np.int32); sts = np.zeros(50, dtype=np.int32)
        hostsim.lib.hostsim_closed_loop(ctypes.byref(p), st.ctypes.data_as(dp), c.ctypes.data_as(dp), 2, 50, warm, ctypes.c_double(mu),
                                        h.ctypes.data_as(dp), it.ctypes.data_as(ip), sts.ctypes.data_as(ip))
        return h, it, sts
    hc, ic, sc = loop(0, 0.0)
    np.testing.assert_allclose(hc, g["out8"], rtol=0, atol=1e-9)
    assert (ic == g["iters"]).all()
    hw, iw, sw = loop(1, 1e-4)
    assert (sw == 0).all()
    np.testing.assert_allclose(hw, g["out8"], rtol=0, atol=1e-6)
    assert iw[0] == ic[0] and iw.sum() < 0.5 * ic.sum()


def test_invalid_numbers_stop_at_the_starting_point(hostsim):
    """NaN / Inf in the state or the coefficients: the reference's Ipopt returns Invalid_Number_Detected (-13) without an
    iteration; so do the C port and both execution shapes of the solver core.  (The reference's binaries, which are
    not part of the repository, are checked too where they are built.)"""
    import oracle_bindings as ob
    g = golden("line_256.npz")
    cases = []
    st = g["states"][0].copy(); st[1] = np.nan; cases.append((st, g["coeffs"][0]))
    st = g["states"][0].copy(); st[3] = np.inf; cases.append((st, g["coeffs"][0]))
    cf = g["coeffs"][0].copy(); cf[0] = np.nan; cases.append((g["states"][0], cf))
    for st, cf in cases:
        if ob.ref_available():
            o = ob.ref_solve(st, cf)
            assert o["status"] == -13 and o["iters"] == 0
        o = ob.port_solve(st, cf)
        assert o["status"] == -13 and o["iters"] == 0
        for mode in (0, 1, 2):
            r = hostsim.solve(st, cf, mode=mode)
            assert r["status"] == -13 and r["iters"] == 0, mode


def test_long_solves_keep_every_filter_entry(hostsim):
    """Extreme initial states (|cte| up to 80 m: objective scaling active, 40-130 iterations at mu = 0.1) grow the filter
    beyond 8 entries; with the filter in its own workspace record (41 entries) the iterates stay Ipopt's: same iteration
    counts and solutions on the thread path, through the per-pass kernels with compaction (the filter entries move with
    the problem) and on the cooperative path."""
    g = golden("long_filter_N25_12.npz")
    for mode in (0, -2, 2):
        same = 0
        for b in range(12):
            r = hostsim.solve(g["states"][b], g["coeffs"][b], mode=mode)
            assert r["status"] == 0
            np.testing.assert_allclose(r["x"], g["x"][b], rtol=0, atol=1e-7)
            assert abs(r["obj"] - g["obj"][b]) <= TOL_OBJ * abs(g["obj"][b])
            same += int(r["iters"] == g["iters"][b])
        assert same >= 11, (mode, same)


@pytest.mark.parametrize("compact", [False, True])
def test_device_memory_layout_on_the_host(hostsim, compact):
    """The device layout (warp-interleaved groups of 32 problems, two regions, slot arithmetic of slot_base() /
    region_doubles(), filter record, per-pass execution, batch compaction into a NaN-poisoned region, guard words behind
    the regions) gives bit-identical results to the one-problem-at-a-time build on a mixed batch of 70 problems (a
    partial last group) that includes long solves, restoration and soft-restoration cases."""
    a, b, c = golden("long_filter_N25_12.npz"), golden("resto_N25_wild_32.npz"), golden("roadmap_256.npz")
    st = np.concatenate([a["states"], b["states"], c["states"][:26]])
    cf = np.concatenate([a["coeffs"], b["coeffs"], c["fit"][:26]])
    r = hostsim.batch_interleaved(st, cf, compact=compact)
    assert r["rc"] == 0, "a write landed outside a workspace region"
    for k in range(len(st)):
        one = hostsim.solve(st[k], cf[k])
        assert r["status"][k] == one["status"] == 0 and r["iters"][k] == one["iters"]
        np.testing.assert_array_equal(r["out8"][k], one["out8"])
        assert r["obj"][k] == one["obj"]


def test_device_memory_layout_on_the_host_long_horizon(hostsim):
    """Same at N = 50, with the problems that take Ipopt's soft restoration steps and its restoration phase."""
    a, b = golden("soft_N50_3.npz"), golden("resto_N50_14.npz")
    st = np.tile(np.concatenate([a["states"], b["states"]]), (3, 1))   # 51 problems: one full group and a partial one
    cf = np.tile(np.concatenate([a["coeffs"], b["coeffs"]]), (3, 1))
    r = hostsim.batch_interleaved(st, cf, compact=True, N=50)
    assert r["rc"] == 0
    for k in range(17):
        one = hostsim.solve(st[k], cf[k], N=50)
        for rep in range(3):
            assert r["status"][k + 17 * rep] == 0 and r["iters"][k + 17 * rep] == one["iters"]
            np.testing.assert_array_equal(r["out8"][k + 17 * rep], one["out8"])


def test_device_memory_layout_with_the_cooperative_finisher(hostsim):
    """As on the device: 14 per-pass rounds with compaction, then the cooperative solver takes every live problem over
    (a failed line search hands a problem to it earlier).  Same solutions as the one-problem cooperative run."""
    a, b = golden("long_filter_N25_12.npz"), golden("resto_N25_wild_32.npz")
    st, cf = np.concatenate([a["states"], b["states"]]), np.concatenate([a["coeffs"], b["coeffs"]])
    ref_x = np.concatenate([a["out8"], b["out8"]])
    r = hostsim.batch_interleaved(st, cf, compact=True, max_rounds=14, coop=True)
    assert r["rc"] == 0 and (r["status"] == 0).all()
    np.testing.assert_allclose(r["out8"], ref_x, rtol=0, atol=1e-6)


def test_filter_reset_heuristic_and_soft_step_after_a_failed_soc(hostsim):
    """Ipopt resets the filter when in 5 successive iterations the last rejected trial point was rejected by the filter
    (IpFilterLSAcceptor.cpp:357-379); ten extreme-state problems where that happens, and one where the line search fails
    right after a failed second-order correction and a soft restoration step follows (the Newton direction is restored
    first).  Same iteration counts and solutions as the reference binaries, on the thread and cooperative paths and in
    the C port (which restates both as well)."""
    import oracle_bindings as ob
    g = golden("rare_paths_N25_11.npz")
    for b in range(11):
        for mode in (0, -2, 2):
            r = hostsim.solve(g["states"][b], g["coeffs"][b], mode=mode)
            assert r["status"] == 0 and r["iters"] == g["iters"][b], (b, mode, r["iters"], g["iters"][b])
            np.testing.assert_allclose(r["x"], g["x"][b], rtol=0, atol=1e-7)
        o = ob.port_solve(g["states"][b], g["coeffs"][b])
        assert o["status"] == 0 and o["iters"] == g["iters"][b]
