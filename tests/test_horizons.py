"""Every horizon the library accepts (b200mpc_create: N in [2, 1024]).  Most kernels change shape with N:
  * the cooperative kernel's lanes run stages t = lane, lane + 32, ... (warp boundaries at N = 32 / 33, 64 / 65);
  * its block holds 4 problems up to N = 51, 3 from 52, 2 from 69, 1 from 103; from N = 205 on it does not fit its
    200 KiB of shared memory and the thread-per-problem kernel finishes the batch instead;
  * the host-buffer transposes of traj (8N-2 fields) and mult (10N-4) tile 128, 32 or 8 problems, or run the wide kernel
    above 2048 fields: traj at N <= 6 / <= 50 / <= 256 / >= 257, mult at N <= 5 / <= 40 / <= 205 / >= 206.
CPU tests hold the host build of the solver core (tests/hostsim) against the C port and its VJP against a dense KKT solve
across horizons; -m gpu runs every execution path of the library at the edge horizons against the host build and the
port, the host-buffer entry points against the device ones, and N = 1024."""
import numpy as np
import pytest

import oracle_bindings as ob
from conftest import golden
from test_sensitivity import PNAMES, _rel, dense_vjp, gbar_of, sens  # noqa: F401  (sens: the VJP fixture)

COOP_MAX_N = 204   # the largest horizon whose cooperative block fits 200 KiB (125 doubles per stage + 10)


def _families(picks):
    """{ncoef: [(state6, coeffs), ...]}: roadmap fits (4), their first three coefficients (3: the same state, since
    cte and epsi are taken at x = 0), line references (2)."""
    g, gl = golden("roadmap_256.npz"), golden("line_256.npz")
    return {4: [(g["states"][b], g["fit"][b]) for b in picks[4]],
            3: [(g["states"][b], g["fit"][b][:3]) for b in picks[3]],
            2: [(gl["states"][b], gl["coeffs"][b]) for b in picks[2]]}


# 8 problems that none of the horizons up to 103 puts on a knife edge
CPU_PICKS = {4: (0, 64, 128), 3: (32, 160), 2: (0, 96, 192)}
# 2 per coefficient count that converge at every horizon up to 1024 (cubic fits of other windows grow like x^3 over the
# few hundred metres of a long horizon and do not)
GPU_PICKS = {4: (0, 100), 3: (100, 200), 2: (37, 100)}


def _worst(d, key, v):
    d[key] = max(d.get(key, 0.0), float(v))


# ------------------------------------------------------------------------------------------------ CPU (host build)
CPU_N = [2, 3, 4, 5, 6, 7, 9, 16, 31, 32, 33, 51, 52, 64, 65, 68, 69, 102, 103, 204, 205]


@pytest.mark.parametrize("N", CPU_N)
def test_host_build_matches_the_port(hostsim, N):
    """Fused loop (mode 0), cooperative solver (2), per-pass with repacking after every pass (-2) and the device memory
    layout with compaction and the cooperative finisher after 4 rounds: the port's status and iteration count exactly,
    the solution within 1e-12 (observed at most 5e-14).  N = 204 / 205 (30 s per port solve): one problem each."""
    fams = _families(CPU_PICKS)
    if N > 103:
        fams = {4: fams[4][:1]} if N % 2 == 0 else {2: fams[2][:1]}
    worst = {}
    for ncoef, probs in fams.items():
        ports = [ob.port_solve(st, cf, params=ob.default_params(N=N)) for st, cf in probs]
        for (st, cf), o in zip(probs, ports):
            assert o["status"] == 0
            for mode in (0, 2, -2):
                h = hostsim.solve(st, cf, mode=mode, N=N)
                assert (h["status"], h["iters"]) == (o["status"], o["iters"]), (ncoef, mode)
                _worst(worst, mode, np.abs(h["x"] - o["x"]).max())
        bi = hostsim.batch_interleaved(np.array([p[0] for p in probs]), np.array([p[1] for p in probs]), compact=True,
                                       max_rounds=4, coop=True, N=N)
        assert bi["rc"] == 0
        np.testing.assert_array_equal(bi["status"], [o["status"] for o in ports])
        np.testing.assert_array_equal(bi["iters"], [o["iters"] for o in ports])
        _worst(worst, "interleaved out8", np.abs(bi["out8"] - np.array([o["out8"] for o in ports])).max())
    print(f"N = {N}: max |host - port| by mode {worst}")
    assert max(worst.values()) < 1e-12, worst


@pytest.mark.parametrize("ncoef", [2, 3, 4])
@pytest.mark.parametrize("N", [2, 3, 5, 10, 33, 50])
def test_host_vjp_matches_the_dense_kkt_solve(sens, N, ncoef):  # noqa: F811
    """hostsim_vjp against the dense KKT solve of test_sensitivity at other horizons and coefficient counts, random
    incoming gradients on out8, traj and obj: within 1e-7 relative to max(1, |grad|).  And the envelope identity
    d obj / d state6 = -lambda at the rows of t = 0."""
    rng = np.random.default_rng(100 * N + ncoef)
    worst = 0.0
    for st, cf in _families(CPU_PICKS)[ncoef][:2]:
        r = sens.solve(st, cf, N=N)
        assert r["status"] == 0
        go8, gt, gob = rng.standard_normal(8), rng.standard_normal(8 * N - 2), float(rng.standard_normal())
        v = sens.vjp(st, cf, r["x"], r["mult"], go8, gt, gob, N=N)
        assert v["status"] == 0
        d = dense_vjp(st, cf, r["x"], r["mult"], gbar_of(go8, gt, N), gob, N=N)
        assert len(v["grad_coeffs"]) == len(d["grad_coeffs"]) == ncoef
        for k in ("grad_state6", "grad_coeffs", "grad_params"):
            worst = max(worst, _rel(v[k], d[k]))
        env = sens.vjp(st, cf, r["x"], r["mult"], None, None, 1.0, N=N)["grad_state6"]
        np.testing.assert_allclose(env, -r["mult"][np.arange(6) * N], rtol=0, atol=1e-12)
    print(f"N = {N}, ncoef = {ncoef}: host build vs dense KKT solve, max relative difference {worst:.2e}")
    assert worst < 1e-7, worst


# ------------------------------------------------------------------------------------------------ GPU
def _on_device(a):
    """(B, K) rows -> a field-major (K, B) CUDA tensor; a 1-D array stays 1-D"""
    import torch
    return torch.as_tensor(np.ascontiguousarray(np.asarray(a).T), device="cuda")


def _solver_kernels(fn):
    """Names of the solver kernels (mpc_*) that run during fn()."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if "mpc_" in e.name and "kernel" in e.name}


def _ran(kernels, name):
    return any(name in k for k in kernels)


EDGE_N = [2, 3, 5, 6, 7, 31, 32, 33, 51, 52, 68, 69, 102, 103, 200, 204, 205, 206, 256, 257]
HANDOVER = 5   # rounds of the per-pass kernels before the finisher takes the rest over
PATHS = {   # name -> (settings, B200MPC_NO_COOP)
    "default": ([], False),   # cooperative kernel for small batches
    "perpass": ([("set_solver_mode", 0, HANDOVER, 0), ("set_compaction", 0.9, 2), ("set_batch_split", 2)], False),
    "fused": ([("set_solver_mode", 1, 0, -1)], False),
    "no_coop": ([], True),
}


@pytest.mark.gpu
@pytest.mark.parametrize("ncoef", [2, 3, 4])
@pytest.mark.parametrize("N", EDGE_N)
def test_every_path_at_the_edge_horizons(hostsim, monkeypatch, N, ncoef):
    """67 problems (2 distinct ones, in every slot of a ragged batch that the split cuts into 64 + 3) on every execution
    path against the host build's matching mode: status and iterations exactly, solution within 1e-9 (FMA contraction
    differs between nvcc and g++); up to N = 103 the same against the C port.  The finisher is the cooperative kernel up
    to N = 204 and the thread-per-problem kernel from N = 205 on, seen in the kernels that ran."""
    import udacitympc_b200 as mp
    probs = _families(GPU_PICKS)[ncoef]
    B = 67
    idx = np.arange(B) % len(probs)
    st = np.array([probs[i][0] for i in idx]); cf = np.array([probs[i][1] for i in idx])
    coop = N <= COOP_MAX_N
    host = {mode: [hostsim.solve(s, c, mode=mode, N=N) for s, c in probs] for mode in (0, 2, -2)}
    bi = hostsim.batch_interleaved(st, cf, compact=True, max_rounds=HANDOVER, coop=coop, N=N)
    ports = [ob.port_solve(s, c, params=ob.default_params(N=N)) for s, c in probs] if N <= 103 else None
    for p in host[0]:
        assert p["status"] == 0
    matching = {"default": 2 if coop else 0, "perpass": -2, "fused": 0, "no_coop": 0}
    worst = {}
    for path, (settings, no_coop) in PATHS.items():
        monkeypatch.setenv("B200MPC_NO_COOP", "1" if no_coop else "0")
        with mp.MPC(device=0, N=N) as m:
            for name, *args in settings:
                getattr(m, name)(*args)
            out = {}
            kernels = _solver_kernels(lambda: out.update(m.solve_batch(st, cf, want_traj=True)))
        finisher_is_coop = coop and path in ("default", "perpass")
        assert _ran(kernels, "mpc_coop_kernel") == finisher_is_coop, (path, kernels)
        assert _ran(kernels, "mpc_fused_kernel") == (not finisher_is_coop), (path, kernels)
        h = host[matching[path]]
        np.testing.assert_array_equal(out["status"], [h[i]["status"] for i in idx], err_msg=path)
        np.testing.assert_array_equal(out["iters"], [h[i]["iters"] for i in idx], err_msg=path)
        _worst(worst, path, np.abs(out["traj"] - np.array([h[i]["x"] for i in idx])).max())
        if path == "perpass":   # the device layout on the host: same compaction and hand-over point
            np.testing.assert_array_equal(out["status"], bi["status"])
            np.testing.assert_array_equal(out["iters"], bi["iters"])
            _worst(worst, "perpass vs interleaved", np.abs(out["out8"] - bi["out8"]).max())
        if ports:
            np.testing.assert_array_equal(out["status"], [ports[i]["status"] for i in idx], err_msg=path)
            np.testing.assert_array_equal(out["iters"], [ports[i]["iters"] for i in idx], err_msg=path)
            _worst(worst, "port", np.abs(out["traj"] - np.array([ports[i]["x"] for i in idx])).max())
    print(f"N = {N}, ncoef = {ncoef}: max |device - reference| {worst}")
    assert max(worst.values()) < 1e-9, worst


def _solve_device(m, st, cf, x_init=None, mult_init=None):
    """solve_batch_warm_device on field-major copies; the results in solve_batch's per-problem layout."""
    import torch
    B, ncoef = cf.shape
    d_st, d_cf = _on_device(st), _on_device(cf)
    d_x = None if x_init is None else _on_device(x_init)
    d_m = None if mult_init is None else _on_device(mult_init)
    o = dict(out8=torch.empty(8, B, dtype=torch.float64, device="cuda"),
             traj=torch.empty(m.num_vars, B, dtype=torch.float64, device="cuda"),
             mult=torch.empty(m.num_mults, B, dtype=torch.float64, device="cuda"),
             cost=torch.empty(B, dtype=torch.float64, device="cuda"),
             status=torch.empty(B, dtype=torch.int32, device="cuda"), iters=torch.empty(B, dtype=torch.int32, device="cuda"))
    torch.cuda.synchronize()   # the call runs on the handle's own stream
    m.solve_batch_warm_device(B, d_st.data_ptr(), d_cf.data_ptr(), ncoef, 0 if d_x is None else d_x.data_ptr(),
                              0 if d_m is None else d_m.data_ptr(), 1e-4, o["out8"].data_ptr(), o["traj"].data_ptr(),
                              o["mult"].data_ptr(), o["cost"].data_ptr(), o["status"].data_ptr(), o["iters"].data_ptr())
    m.wait()
    return {k: v.cpu().numpy().T for k, v in o.items()}


def _vjp_device(m, st, cf, traj, mult, go8, gt, gob):
    import torch
    B, ncoef = cf.shape
    ins = [_on_device(a) for a in (st, cf, traj, mult, go8, gt, gob)]
    gs, gc, gp = (torch.empty(k, B, dtype=torch.float64, device="cuda") for k in (6, ncoef, 8))
    status = torch.empty(B, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    m.solve_batch_vjp_device(B, ins[0].data_ptr(), ins[1].data_ptr(), ncoef, *[t.data_ptr() for t in ins[2:]],
                             gs.data_ptr(), gc.data_ptr(), gp.data_ptr(), status.data_ptr())
    m.wait()
    return dict(grad_state6=gs.cpu().numpy().T, grad_coeffs=gc.cpu().numpy().T, grad_params=gp.cpu().numpy().T,
                status=status.cpu().numpy())


def _assert_same(h, d, keys, what):
    for k in keys:
        np.testing.assert_array_equal(h[k], d[k], err_msg=f"{what}: {k}")


@pytest.mark.gpu
@pytest.mark.parametrize("N", [5, 6, 7, 40, 41, 50, 51, 205, 206, 256, 257])
def test_host_buffer_entries_equal_the_device_entries_bitwise(N):
    """traj, mult, x_init, mult_init and g_traj of the host-buffer entry points go through the tiled transposes (or the
    wide kernel); the device entry points take field-major buffers as they are.  Both give the same bits, on batches
    whose last tile is partial for every tile size: a cold solve with traj and mult out, a warm start from its shifted
    solution and a perturbed state, and the VJP at the cold solution."""
    import udacitympc_b200 as mp
    from udacitympc_b200 import synth
    st_all, cf_all = synth.line_problems(1000)
    rng = np.random.default_rng(N)
    with mp.MPC(device=0, N=N, max_iter=400) as m:
        for B in (1, 7, 9, 33, 129, 1000):
            st, cf = st_all[:B], cf_all[:B]
            h = m.solve_batch(st, cf, want_traj=True, want_mult=True)
            ok = h["status"] == 0   # at N >= 256 one problem of the first 33 needs more than 400 iterations
            assert ok.mean() > 0.9, (B, h["status"])
            _assert_same(h, _solve_device(m, st, cf), ("out8", "traj", "mult", "cost", "status", "iters"), f"cold B={B}")
            x0, m0 = mp.shift_solution(h["traj"], h["mult"], N)
            st2 = st.copy()
            st2[:, 3] += 0.5
            w = m.solve_batch(st2, cf, want_traj=True, want_mult=True, x_init=x0, mult_init=m0)
            assert (w["status"][ok] == 0).all() and (w["iters"] > 0).all()
            _assert_same(w, _solve_device(m, st2, cf, x0, m0), ("out8", "traj", "mult", "cost", "status", "iters"),
                         f"warm B={B}")
            go8, gt, gob = rng.standard_normal((B, 8)), rng.standard_normal((B, m.num_vars)), rng.standard_normal(B)
            v = m.solve_batch_vjp(st, cf, h["traj"], h["mult"], go8, gt, gob, want_params=True)
            assert (v["status"][ok] == 0).all()
            _assert_same(v, _vjp_device(m, st, cf, h["traj"], h["mult"], go8, gt, gob),
                         ("grad_state6", "grad_coeffs", "grad_params", "status"), f"vjp B={B}")


@pytest.mark.gpu
@pytest.mark.parametrize("N", [2, 3, 33, 69, 205])
def test_device_vjp_matches_the_host_build_at_edge_horizons(sens, N):  # noqa: F811
    """The device VJP against hostsim_vjp for every coefficient count, random incoming gradients; at N = 33 also with
    per-problem costs (cost8).  Within 1e-8 relative to max(1, |grad|)."""
    import udacitympc_b200 as mp
    rng = np.random.default_rng(N)
    worst = 0.0
    with mp.MPC(device=0, N=N) as m:
        for ncoef, probs in _families(GPU_PICKS).items():
            st, cf = np.array([p[0] for p in probs]), np.array([p[1] for p in probs])
            B = len(st)
            # per-problem costs: ref_v, then the seven weights
            for cost in ([None, np.c_[rng.uniform(30.0, 45.0, B), rng.uniform(0.5, 2.0, (B, 7))]] if N == 33 else [None]):
                r = m.solve_batch(st, cf, want_traj=True, want_mult=True, cost_params=cost)
                assert (r["status"] == 0).all(), (ncoef, r["status"])
                go8, gt, gob = rng.standard_normal((B, 8)), rng.standard_normal((B, m.num_vars)), rng.standard_normal(B)
                v = m.solve_batch_vjp(st, cf, r["traj"], r["mult"], go8, gt, gob, want_params=True, cost_params=cost)
                for b in range(B):
                    params = {} if cost is None else dict(zip(PNAMES, cost[b]))
                    h = sens.vjp(st[b], cf[b], r["traj"][b], r["mult"][b], go8[b], gt[b], gob[b], N=N, **params)
                    assert v["status"][b] == h["status"] == 0, (ncoef, b)
                    for k in ("grad_state6", "grad_coeffs", "grad_params"):
                        worst = max(worst, _rel(v[k][b], h[k]))
    print(f"N = {N}: device vs host build VJP, max relative difference {worst:.2e}")
    assert worst < 1e-8, worst


@pytest.mark.gpu
def test_the_longest_horizon(hostsim):
    """N = 1024 (the transposes at their largest K, the thread finisher): three problems on the default path and on
    per-pass kernels against the host build, and the size-independent properties: the bounds hold, rolling the model
    with the solution's actuators reproduces its states, both launch sequences give the same answer."""
    import udacitympc_b200 as mp
    N = 1024
    g, gl = golden("roadmap_256.npz"), golden("line_256.npz")
    st = np.array([g["states"][200], gl["states"][37], gl["states"][100]])
    cf = np.array([g["fit"][200], np.r_[gl["coeffs"][37], 0, 0], np.r_[gl["coeffs"][100], 0, 0]])
    with mp.MPC(device=0, N=N, max_iter=400) as m:
        r = m.solve_batch(st, cf, want_traj=True, want_mult=True)
        m.set_solver_mode(0, 12, 0)
        r2 = m.solve_batch(st, cf, want_traj=True, want_mult=True)
    worst = 0.0
    for b in range(3):
        h = hostsim.solve(st[b], cf[b], N=N, max_iter=400)
        assert h["status"] == r["status"][b] == 0 and h["iters"] == r["iters"][b], b
        worst = max(worst, np.abs(r["traj"][b] - h["x"]).max())
    print(f"N = 1024: max |device - host build| {worst:.2e}, iterations {r['iters']}")
    assert worst < 1e-9, worst
    np.testing.assert_array_equal(r["status"], r2["status"])
    np.testing.assert_array_equal(r["iters"], r2["iters"])
    np.testing.assert_allclose(r2["traj"], r["traj"], rtol=0, atol=1e-9)
    T = r["traj"]
    DEL, ACC = T[:, 6 * N:7 * N - 1], T[:, 7 * N - 1:]
    assert np.abs(DEL).max() <= 0.436332 and np.abs(ACC).max() <= 1.0
    np.testing.assert_allclose(T[:, [0, N, 2 * N, 3 * N, 4 * N, 5 * N]], st, rtol=0, atol=1e-12)
    with mp.MPC(device=0) as m0:
        roll = mp.rollout_batch(st[:, :4], np.stack([DEL, ACC], axis=2), 0.05, 2.67, mpc=m0)
    err = np.abs(np.stack([T[:, 1:N], T[:, N + 1:2 * N], T[:, 2 * N + 1:3 * N], T[:, 3 * N + 1:4 * N]], axis=2) - roll).max()
    assert err < 1e-4, err
