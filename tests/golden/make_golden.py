"""Generates the golden fixtures in this directory by running THE REFERENCE ITSELF in the build container:
  * oracle/_ref/libmpc_ref.so      the reference's prebuilt Ipopt 3.12.7 + MUMPS 4.10.0 binaries driven on the NLP of
                                   mpc_to_line/solution/MPC.cpp (default options + print_level 0)
  * oracle/_ref/libhelpers_ref.so  the reference's polyfit / polyeval / globalKinematic compiled from where they lie
and extracts the roadmap centre line (mpc_to_line/roadmap.csv columns 4,5) as an input data fixture.

    python tests/golden/make_golden.py        (needs /root/reference; `make -C oracle` first)

The fixtures are small .npz files; tests never read /root/reference.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)

import oracle_bindings as ob  # noqa: E402

REF = os.environ.get("REFERENCE_ROOT", "/root/reference")


def write_centerline():
    rm = np.loadtxt(os.path.join(REF, "mpc_to_line", "roadmap.csv"), delimiter=",")
    out = os.path.join(ROOT, "udacitympc_b200", "data")
    os.makedirs(out, exist_ok=True)
    with open(os.path.join(out, "roadmap_centerline.csv"), "w") as f:
        for x, y in rm[:, 4:6]:
            f.write(f"{float(x)!r},{float(y)!r}\n")
    # the whole file in the reference's own 7-column format (left edge x,y, right edge x,y, centre x,y, slope): the input
    # of the library's reader b200mpc_read_roadmap_csv
    with open(os.path.join(out, "roadmap.csv"), "w") as f:
        for row in rm:
            f.write(",".join(repr(float(v)) for v in row) + "\n")


def solve_set(states, coeffs, **kw):
    B = len(states)
    N = kw.get("N", 25)
    out8 = np.zeros((B, 8)); x = np.zeros((B, 8 * N - 2)); obj = np.zeros(B)
    st = np.zeros(B, dtype=np.int32); it = np.zeros(B, dtype=np.int32); resto = np.zeros(B, dtype=np.int32)
    regu = np.zeros(B); lsmax = np.zeros(B, dtype=np.int32)
    for b in range(B):
        r = ob.ref_solve(states[b], coeffs[b], trace=True, **kw)   # kw: N, dt, Lf, ref_v, delta_max, a_max, weights
        out8[b] = r["out8"]; x[b] = r["x"]; obj[b] = r["obj"]; st[b] = r["status"]; it[b] = r["iters"]
        tr = r["trace"]
        resto[b] = int((tr[:, 9] >= 100).any())
        regu[b] = tr[:, 6].max()
        lsmax[b] = int((tr[:, 9] % 100).max())
    return dict(out8=out8, x=x, obj=obj, status=st, iters=it, used_restoration=resto, max_regu=regu, max_ls_trials=lsmax)


def main():
    from udacitympc_b200 import synth
    write_centerline()

    # ---- config 1: solution/main.cpp closed loop, 50 steps
    coeffs = ob.ref_polyfit([-100.0, 100.0], [-1.0, -1.0], 1)
    x, y, psi, v = -1.0, 10.0, 0.0, 10.0
    cte = ob.ref_polyeval(coeffs, x) - y
    epsi = psi - np.arctan(coeffs[1])
    state = np.array([x, y, psi, v, cte, epsi])
    rows8, rowsx, cost, iters, states = [], [], [], [], []
    for _ in range(50):
        states.append(state.copy())
        r = ob.ref_solve(state, coeffs)
        assert r["status"] == 0
        rows8.append(r["out8"].copy()); rowsx.append(r["x"].copy()); cost.append(r["obj"]); iters.append(r["iters"])
        state = r["out8"][:6].copy()
    np.savez_compressed(os.path.join(HERE, "config1_closed_loop.npz"), coeffs=coeffs, states=np.array(states),
                        out8=np.array(rows8), x=np.array(rowsx), cost=np.array(cost), iters=np.array(iters, dtype=np.int32))

    # ---- config 3 slice: 256 randomized degree-1 problems
    st, cf = synth.line_problems(256)
    np.savez_compressed(os.path.join(HERE, "line_256.npz"), states=st, coeffs=cf, **solve_set(st, cf))

    # ---- config 2(ii) + 4 slice: 256 roadmap windows, reference polyfit (degree 3), then degree-3 MPC
    xs, ys = synth.roadmap_windows(256)
    fit = np.array([ob.ref_polyfit(xs[b], ys[b], 3) for b in range(256)])
    st3 = synth.roadmap_problems(256, fit)
    np.savez_compressed(os.path.join(HERE, "roadmap_256.npz"), xs=xs, ys=ys, fit=fit, states=st3, **solve_set(st3, fit))

    # ---- other horizons (degree 3): N=10 and N=50, 64 problems each
    for N in (10, 50):
        np.savez_compressed(os.path.join(HERE, f"roadmap_N{N}_64.npz"), states=st3[:64], coeffs=fit[:64],
                            **solve_set(st3[:64], fit[:64], N=N))

    # ---- non-default parameters (weights, bounds, Lf, dt, ref_v) through the same reference binaries is not
    # possible: the TNLP restates MPC.cpp with unit weights.  Lf/dt/ref_v/bounds ARE parameters of it:
    kw = dict(N=20, dt=0.08, Lf=2.0, ref_v=25.0, delta_max=0.3, a_max=0.7)
    np.savez_compressed(os.path.join(HERE, "line_params_64.npz"), states=st[:64], coeffs=cf[:64],
                        params=np.array([kw["N"], kw["dt"], kw["Lf"], kw["ref_v"], kw["delta_max"], kw["a_max"]]),
                        **solve_set(st[:64], cf[:64], **kw))

    # ---- config 2(i): bicycle steps with the reference's globalKinematic (dt=0.3, Lf=2) and 25-step rollouts
    ks, ka = synth.kinematic_inputs(256, H=25)
    one = np.array([ob.ref_kinematic(ks[b], ka[b, 0], 0.3) for b in range(256)])
    roll = np.zeros((256, 25, 4))
    for b in range(256):
        s = ks[b].copy()
        for h in range(25):
            s = ob.ref_kinematic(s, ka[b, h], 0.3)
            roll[b, h] = s
    np.savez_compressed(os.path.join(HERE, "kinematic_256.npz"), states=ks, act=ka, one_step=one, rollout=roll)

    # ---- polyfit on other shapes with the reference's helpers.h
    rng = np.random.default_rng(7)
    shapes = {}
    for (m, order) in [(2, 1), (3, 2), (4, 3), (6, 1), (6, 2), (6, 3), (8, 3), (7, 4), (12, 5)]:
        px = np.sort(rng.uniform(-3, 3, size=(32, m)), axis=1)
        py = rng.uniform(-2, 2, size=(32, m))
        shapes[f"xs_{m}_{order}"] = px
        shapes[f"ys_{m}_{order}"] = py
        shapes[f"fit_{m}_{order}"] = np.array([ob.ref_polyfit(px[b], py[b], order) for b in range(32)])
    np.savez_compressed(os.path.join(HERE, "polyfit_shapes.npz"), **shapes)
    print("golden fixtures written to", HERE)


if __name__ == "__main__" and not {"--config3", "--n100", "--resto", "--soft", "--long-filter", "--rare-paths", "--weights", "--frontend", "--loops"} & set(sys.argv):
    main()


def weights():
    """Non-unit cost weights through the reference binaries: the TNLP's seven weights (oracle/ref_build/mpc_tnlp.cpp,
    ref_mpc_solve_w) multiply the seven terms MPC.cpp:57-76 adds with weight 1.  Two weight sets x (32 degree-1 problems
    + 32 degree-3 roadmap problems)."""
    from udacitympc_b200 import synth
    st, cf = synth.line_problems(32)
    g = np.load(os.path.join(HERE, "roadmap_256.npz"))
    sets = {"a": [3.0, 0.5, 0.2, 10.0, 2.0, 50.0, 4.0], "b": [2000.0, 2000.0, 1.0, 5.0, 5.0, 200.0, 10.0]}
    out = dict(line_states=st, line_coeffs=cf, road_states=g["states"][:32], road_coeffs=g["fit"][:32])
    for name, w in sets.items():
        out[f"w_{name}"] = np.array(w)
        for kind, (s_, c_) in (("line", (st, cf)), ("road", (g["states"][:32], g["fit"][:32]))):
            r = solve_set(s_, c_, weights=w)
            for k, v in r.items():
                out[f"{kind}_{name}_{k}"] = v
    np.savez_compressed(os.path.join(HERE, "weights_64.npz"), **out)
    print({k: int(out[k].sum()) for k in out if k.endswith("used_restoration")}, {k: out[k].tolist() for k in out if k.endswith("_status")})


if __name__ == "__main__" and "--weights" in sys.argv:
    weights()


def frontend():
    """Roadmap front-end fixture (SURVEY 8f2): what produces (coeffs, cte, epsi) in front of MPC::Solve.  Built from the
    reference's own pieces where they run: its roadmap.csv (columns 4, 5 = centre line, custom_MPC.cpp:206-211), the
    nearest-centre-line-point rule of custom_MPC.cpp:177-185 (squared distance, first minimum = ind[0] of CppAD::index_sort),
    the global -> vehicle frame transform, the reference's OWN polyfit (helpers.h:24-44, oracle/_ref/libhelpers_ref.so)
    on the 6 waypoints from there, and cte = polyeval(coeffs, 0) - 0, epsi = 0 - atan(coeffs[1]) as solution/main.cpp:34-37
    defines them.  custom_MPC.cpp itself cannot run (CppAD absent, hard-coded /home/honda path, file name parsed as file
    content), so the selection rule and the frame change are restated here in numpy, the fit is the reference's."""
    rm = np.loadtxt(os.path.join(REF, "mpc_to_line", "roadmap.csv"), delimiter=",")
    cl = rm[:, 4:6]
    rng = np.random.default_rng(20240607)
    B = 256
    idx = rng.integers(0, len(cl) - 1, size=B)
    tng = cl[idx + 1] - cl[idx]
    ang = np.arctan2(tng[:, 1], tng[:, 0])
    nrm = np.stack([-np.sin(ang), np.cos(ang)], axis=1)
    frac = rng.uniform(0, 1, size=B)[:, None]
    pos = cl[idx] + frac * tng + rng.uniform(-3.0, 3.0, size=B)[:, None] * nrm
    psi = ang + rng.uniform(-0.4, 0.4, size=B)
    v = rng.uniform(3.0, 35.0, size=B)
    poses = np.column_stack([pos, psi, v])
    # a few poses far from the road and next to its end (window clamped to the last 6 points)
    poses[0, :2] = cl[-1] + [1.0, 2.0]; poses[1, :2] = cl[-3] + [0.5, -0.5]; poses[2, :2] = cl[0] - [20.0, 5.0]
    state6 = np.zeros((B, 6)); coeffs = np.zeros((B, 4)); nearest = np.zeros(B, dtype=np.int32)
    for b in range(B):
        x, y, p = poses[b, 0], poses[b, 1], poses[b, 2]
        d = (x - cl[:, 0]) * (x - cl[:, 0]) + (y - cl[:, 1]) * (y - cl[:, 1])
        i0 = int(np.argmin(d))   # first minimum
        nearest[b] = i0
        i0 = min(i0, len(cl) - 6)
        dx, dy = cl[i0:i0 + 6, 0] - x, cl[i0:i0 + 6, 1] - y
        lx = np.cos(p) * dx + np.sin(p) * dy
        ly = np.cos(p) * dy - np.sin(p) * dx
        c = ob.ref_polyfit(lx, ly, 3)
        coeffs[b] = c
        state6[b] = [0.0, 0.0, 0.0, poses[b, 3], ob.ref_polyeval(c, 0.0) - 0.0, 0.0 - np.arctan(c[1])]
    np.savez_compressed(os.path.join(HERE, "frontend_256.npz"), poses=poses, centerline=cl, state6=state6, coeffs=coeffs, nearest=nearest)
    print("frontend fixture:", B, "poses, nearest index range", nearest.min(), nearest.max())


if __name__ == "__main__" and "--frontend" in sys.argv:
    write_centerline()
    frontend()


def config3():
    """BASELINE configs[2]: 4096 randomized degree-1 problems (SURVEY 8d config 3), solved by the reference binaries
    on all cores.  Only the returned 8-vector, objective, status and iteration count are stored (the full 198-vector
    of the first 256 problems is in line_256.npz)."""
    import multiprocessing as mp
    from udacitympc_b200 import synth
    st, cf = synth.line_problems(4096)
    with mp.get_context("fork").Pool(os.cpu_count()) as pool:
        res = pool.map(_solve_one, [(st[b], cf[b]) for b in range(4096)], chunksize=64)
    np.savez_compressed(os.path.join(HERE, "config3_line_4096.npz"), out8=np.array([r[0] for r in res]),
                        obj=np.array([r[1] for r in res]), status=np.array([r[2] for r in res], dtype=np.int32),
                        iters=np.array([r[3] for r in res], dtype=np.int32), used_restoration=np.array([r[4] for r in res], dtype=np.int32))


def _solve_one(a):
    r = ob.ref_solve(a[0], a[1], trace=True)
    return r["out8"], r["obj"], r["status"], r["iters"], int((r["trace"][:, 9] >= 100).any())


if __name__ == "__main__" and "--config3" in sys.argv:
    config3()


def n100():
    """BASELINE configs[4] at its longest horizon: the first 64 roadmap problems with N=100 (same inputs as
    roadmap_N{10,50}_64.npz)."""
    g = np.load(os.path.join(HERE, "roadmap_256.npz"))
    st3, fit = g["states"], g["fit"]
    np.savez_compressed(os.path.join(HERE, "roadmap_N100_64.npz"), states=st3[:64], coeffs=fit[:64],
                        **solve_set(st3[:64], fit[:64], N=100))


if __name__ == "__main__" and "--n100" in sys.argv:
    n100()


def _solve_resto(a):
    r = ob.ref_solve(a[0], a[1], N=a[2], trace=True)
    return r["out8"], r["obj"], r["status"], r["iters"], int((r["trace"][:, 9] >= 100).any()), r["x"]


def resto():
    """Problems on which the reference's Ipopt entered its restoration phase: the first 48 such problems among 8192
    random roadmap problems at N=100, all 14 among 65 536 at N=50, and the first 32 among 32 768 at the reference's own
    N=25 with initial states far outside the benchmark distribution (lateral offset +-20 m, heading error +-1.5 rad,
    speed 1..60 m/s; 346 of them use it).  Inputs: synth.roadmap_windows / roadmap_problems with the seeds below; the
    fit is numpy's least-squares fit of the window.  Takes ~5 min on 8 cores."""
    import multiprocessing as mp
    from udacitympc_b200 import synth
    for N, n, keep, wild in ((100, 8192, 48, False), (50, 65536, 14, False), (25, 32768, 32, True)):
        xs, ys = synth.roadmap_windows(n, synth.MT19937_64(878))
        V = np.stack([xs ** i for i in range(4)], axis=2)
        fit = np.stack([np.linalg.lstsq(V[b], ys[b], rcond=None)[0] for b in range(n)])
        st = synth.roadmap_problems(n, fit, synth.MT19937_64(879))
        if wild:
            u = synth.MT19937_64(880).uniform(3 * n).reshape(n, 3)
            y = -20.0 + 40.0 * u[:, 0]
            psi = np.arctan(fit[:, 1]) - 1.5 + 3.0 * u[:, 1]
            v = 1.0 + 59.0 * u[:, 2]
            st = np.ascontiguousarray(np.stack([np.zeros(n), y, psi, v, fit[:, 0] - y, psi - np.arctan(fit[:, 1])], axis=1))
        with mp.get_context("fork").Pool(os.cpu_count()) as pool:
            res = pool.map(_solve_resto, [(st[b], fit[b], N) for b in range(n)], chunksize=8)
        sel = [b for b in range(n) if res[b][4] and res[b][2] == 0][:keep]
        name = f"resto_N{N}_{'wild_' if wild else ''}{len(sel)}.npz"
        np.savez_compressed(os.path.join(HERE, name), index=np.array(sel, dtype=np.int32),
                            states=st[sel], coeffs=fit[sel], out8=np.array([res[b][0] for b in sel]),
                            obj=np.array([res[b][1] for b in sel]), iters=np.array([res[b][3] for b in sel], dtype=np.int32),
                            x=np.array([res[b][5] for b in sel]).astype(np.float64), n_problems=n,
                            n_used_restoration=int(sum(r[4] for r in res)))
        print(f"N={N}{' wild' if wild else ''}: {int(sum(r[4] for r in res))} of {n} problems used the restoration phase; kept {len(sel)}")


if __name__ == "__main__" and "--resto" in sys.argv:
    resto()


def soft():
    """Problems on which the reference's Ipopt takes soft-restoration steps ('s' / 'S' in its iteration log) and never
    enters the restoration phase proper: #1606, #7262, #14731 of the 16 384 wild N=50 problems (same generator and seeds
    as resto(); found with tools/resto_campaign.py 50 16384 --wild as the iteration-count mismatches of mode 1 that
    vanish in mode 2)."""
    from udacitympc_b200 import synth
    n, N, sel = 16384, 50, [1606, 7262, 14731]
    xs, ys = synth.roadmap_windows(n, synth.MT19937_64(878))
    V = np.stack([xs ** i for i in range(4)], axis=2)
    fit = np.stack([np.linalg.lstsq(V[b], ys[b], rcond=None)[0] for b in range(n)])
    u = synth.MT19937_64(880).uniform(3 * n).reshape(n, 3)
    y = -20.0 + 40.0 * u[:, 0]
    psi = np.arctan(fit[:, 1]) - 1.5 + 3.0 * u[:, 1]
    v = 1.0 + 59.0 * u[:, 2]
    st = np.ascontiguousarray(np.stack([np.zeros(n), y, psi, v, fit[:, 0] - y, psi - np.arctan(fit[:, 1])], axis=1))
    res = [_solve_resto((st[b], fit[b], N)) for b in sel]
    assert all(r[2] == 0 and r[4] == 0 for r in res)
    np.savez_compressed(os.path.join(HERE, "soft_N50_3.npz"), index=np.array(sel, dtype=np.int32), states=st[sel], coeffs=fit[sel],
                        out8=np.array([r[0] for r in res]), obj=np.array([r[1] for r in res]),
                        iters=np.array([r[3] for r in res], dtype=np.int32), x=np.array([r[5] for r in res]))


if __name__ == "__main__" and "--soft" in sys.argv:
    soft()


def long_filter():
    """Long solves from extreme initial states (lateral offset up to +-80 m, heading error +-3 rad, 0.1..80 m/s: the
    |cte| > 50 objective-scaling branch) whose filter grows beyond 8 entries: 12 of the 32 768 "wilder" N=25 problems of
    tools/resto_campaign.py that the reference solves without its restoration phase."""
    from udacitympc_b200 import synth
    n, N, sel = 32768, 25, [82, 505, 1535, 1543, 1606, 1612, 1870, 2957, 3534, 3666, 4014, 4418]
    if "--rare-paths" in sys.argv:
        # filter reset heuristic (IpFilterLSAcceptor.cpp:357-379) active: the first ten; a soft restoration step right
        # after a failed second-order correction: #15085
        sel = [5000, 8393, 11169, 14810, 17473, 19085, 22428, 31634, 31855, 32637, 15085]
    xs, ys = synth.roadmap_windows(n, synth.MT19937_64(878))
    V = np.stack([xs ** i for i in range(4)], axis=2)
    fit = np.stack([np.linalg.lstsq(V[b], ys[b], rcond=None)[0] for b in range(n)])
    u = synth.MT19937_64(880).uniform(3 * n).reshape(n, 3)
    y = -80.0 + 160.0 * u[:, 0]
    psi = np.arctan(fit[:, 1]) - 3.0 + 6.0 * u[:, 1]
    v = 0.1 + 79.9 * u[:, 2]
    st = np.ascontiguousarray(np.stack([np.zeros(n), y, psi, v, fit[:, 0] - y, psi - np.arctan(fit[:, 1])], axis=1))
    res = [_solve_resto((st[b], fit[b], N)) for b in sel]
    assert all(r[2] == 0 and r[4] == 0 for r in res)
    np.savez_compressed(os.path.join(HERE, "rare_paths_N25_11.npz" if "--rare-paths" in sys.argv else "long_filter_N25_12.npz"),
                        index=np.array(sel, dtype=np.int32), states=st[sel],
                        coeffs=fit[sel], out8=np.array([r[0] for r in res]), obj=np.array([r[1] for r in res]),
                        iters=np.array([r[3] for r in res], dtype=np.int32), x=np.array([r[5] for r in res]))


if __name__ == "__main__" and ("--long-filter" in sys.argv or "--rare-paths" in sys.argv):
    long_filter()


def _solver():
    """The reference's binaries when they are built (oracle/_ref), else the C restatement of its algorithm
    (oracle/libmpc_oracle.so), which reproduces the reference's iterates on the fixtures above."""
    return ("reference", ob.ref_solve) if ob.ref_available() else ("port", ob.port_solve)


def loops():
    """Fixtures of two GPU tests that solve one problem at a time on the CPU and compare:
      * roadmap_closed_loop_12x8.npz: solution/main.cpp:51-76 for 12 vehicles of roadmap_256.npz (every 20th), 8 steps,
        each step starting from the state the previous solve predicted;
      * straggler_set3.npz: the problem with the most interior-point iterations (68) of bench.py's input set 3
        (synth.SEED + 3000 / 3001, 65 536 roadmap problems), index 31134."""
    from udacitympc_b200 import synth
    src, solve = _solver()
    g = np.load(os.path.join(HERE, "roadmap_256.npz"))
    sel = np.arange(0, 240, 20)
    K, J = 8, len(sel)
    out8 = np.zeros((K, J, 8)); obj = np.zeros((K, J)); st = np.zeros((K, J), dtype=np.int32); it = np.zeros((K, J), dtype=np.int32)
    for j, b in enumerate(sel):
        s = g["states"][b].copy()
        for k in range(K):
            r = solve(s, g["fit"][b])
            out8[k, j], obj[k, j], st[k, j], it[k, j] = r["out8"], r["obj"], r["status"], r["iters"]
            s = r["out8"][:6].copy()
    # the first step is a problem of roadmap_256.npz: the solver used here must reproduce the reference's result there
    assert (it[0] == g["iters"][sel]).all() and np.abs(out8[0] - g["out8"][sel]).max() < 1e-9
    np.savez_compressed(os.path.join(HERE, "roadmap_closed_loop_12x8.npz"), index=sel, out8=out8, obj=obj, status=st, iters=it,
                        source=np.array(src))
    B, j = 65536, 31134
    xs, ys = synth.roadmap_windows(B, synth.MT19937_64(synth.SEED + 3000))
    fit = ob.port_polyfit(xs[j], ys[j], 3)
    state = synth.roadmap_problems(B, np.tile(fit, (B, 1)), synth.MT19937_64(synth.SEED + 3001))[j]
    r = solve(state, fit)
    np.savez_compressed(os.path.join(HERE, "straggler_set3.npz"), index=j, state=state, coeffs=fit, x=r["x"], out8=r["out8"], obj=r["obj"],
                        status=r["status"], iters=r["iters"], source=np.array(src))
    print(src, "loop iterations", it.sum(), "straggler", r["status"], r["iters"])


if __name__ == "__main__" and "--loops" in sys.argv:
    loops()
