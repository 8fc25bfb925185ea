#!/usr/bin/env python
"""Cost of the forward sensitivities against the solve and the adjoint sensitivities, on bench.py's workload (65 536
seeded roadmap problems, degree-3 fits, N = 25).  Three arms on device buffers, timed with CUDA events and alternated over
--reps repetitions:
    solve  solve_batch_warm_device from the default start point (x_init = NULL), returning traj and mult
    vjp    solve_batch_vjp_model_device at that solution, incoming gradients on out8, traj and obj, every gradient out
    jvp    solve_batch_jvp_device at that solution, tangents of all four input groups, t_out8, t_traj and t_obj out
and the latency of a lone caller's one-problem JVP through host buffers (solve_batch_jvp).  Also the bytes the JVP
kernel moves (its inputs, outputs and the workspace rows of its sweeps), as a bound on its time.  Prints one JSON line,
with the card's name and power limit read in the same run.
    python tools/jvp_bench.py [--batch 65536] [--reps 5] [--lone 200]"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from vjp_bench import card  # noqa: E402


def jvp_bytes(B, N, ncoef=4):
    """Bytes the JVP must move at least: inputs (state6, coeffs, traj, mult and the tangents: 6 + ncoef + 8 + 4), outputs
    (t_out8, t_traj, t_obj, status) and the workspace traffic of its sweeps (load: 22 rows per stage written; right-hand
    sides: 22 read, 14 written; factor: 22 + 6 + 8 read, 13 written; roll-out: 13 + 12 + 6 read, 8 written; outputs: 8
    read)."""
    M = N - 1
    io = 6 + ncoef + (8 * N - 2) + (10 * N - 4) + 6 + ncoef + 8 + 4 + 8 + (8 * N - 2) + 1 + 0.5
    ws = N * (22 + 22 + 14 + 36 + 13 + 31 + 8 + 8) + M * 2
    return 8.0 * B * (io + ws)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--lone", type=int, default=200)
    a = ap.parse_args()
    import torch
    import bench
    import udacitympc_b200 as mp
    if not torch.cuda.is_available():
        raise SystemExit("jvp_bench.py needs a CUDA device")
    B, N = a.batch, 25
    dev = torch.device("cuda:0")
    m = mp.MPC(device=0)
    st, cf = bench.make_workload("roadmap", B, mpc=m)
    nv, nm = m.num_vars, m.num_mults
    T = lambda x: torch.from_numpy(np.ascontiguousarray(x.T)).to(dev)
    dst, dcf = T(st), T(cf)
    E = lambda *s: torch.empty(s, dtype=torch.float64, device=dev)
    out8, traj, mult, obj = E(8, B), E(nv, B), E(nm, B), E(B)
    status, vstatus, jstatus = (torch.empty(B, dtype=torch.int32, device=dev) for _ in range(3))
    rng = np.random.default_rng(0)
    g8, gt, go = T(rng.standard_normal((B, 8))), T(rng.standard_normal((B, nv))), torch.from_numpy(rng.standard_normal(B)).to(dev)
    gs, gc, gp, gm = E(6, B), E(4, B), E(8, B), E(4, B)
    from udacitympc_b200.api import default_params
    p = default_params()
    p8 = np.array([getattr(p, k) for k in mp.PARAM_NAMES]); m4 = np.array([getattr(p, k) for k in mp.MODEL_NAMES])
    t6, tc = T(rng.standard_normal((B, 6))), T(rng.standard_normal((B, 4)) * np.array([1e-1, 1e-2, 1e-4, 1e-6]))
    t8, tm = T(rng.standard_normal((B, 8)) * p8), T(rng.standard_normal((B, 4)) * m4)
    to8, tt, tob = E(8, B), E(nv, B), E(B)
    ts = torch.cuda.Stream()
    torch.cuda.synchronize()   # the inputs were written on the default stream
    torch.cuda.set_stream(ts)
    s = ts.cuda_stream

    def solve():
        m.solve_batch_warm_device(B, dst.data_ptr(), dcf.data_ptr(), 4, 0, 0, 0.0, out8.data_ptr(), traj.data_ptr(),
                                  mult.data_ptr(), obj.data_ptr(), status.data_ptr(), 0, s)

    def vjp():
        m.solve_batch_vjp_model_device(B, dst.data_ptr(), dcf.data_ptr(), 4, 0, 0, traj.data_ptr(), mult.data_ptr(),
                                       g8.data_ptr(), gt.data_ptr(), go.data_ptr(), gs.data_ptr(), gc.data_ptr(),
                                       gp.data_ptr(), gm.data_ptr(), vstatus.data_ptr(), s)

    def jvp():
        m.solve_batch_jvp_device(B, dst.data_ptr(), dcf.data_ptr(), 4, 0, 0, traj.data_ptr(), mult.data_ptr(), t6.data_ptr(),
                                 tc.data_ptr(), t8.data_ptr(), tm.data_ptr(), to8.data_ptr(), tt.data_ptr(), tob.data_ptr(),
                                 jstatus.data_ptr(), s)

    def timed(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(ts)
        for _ in range(n):
            fn()
        e1.record(ts)
        e1.synchronize()
        return e0.elapsed_time(e1) / n

    solve(); vjp(); jvp(); solve(); vjp(); jvp()   # warm-up: modules, solve graph, workspace
    torch.cuda.synchronize()
    t_solve, t_vjp, t_jvp = [], [], []
    for _ in range(a.reps):
        t_solve.append(timed(solve, 3))
        t_vjp.append(timed(vjp, 10))
        t_jvp.append(timed(jvp, 10))
    st_h = status.cpu().numpy()
    conv = (st_h == 0) | (st_h == 1)
    jst = jstatus.cpu().numpy()
    finite = bool(np.isfinite(to8.cpu().numpy()[:, conv]).all() and np.isfinite(tt.cpu().numpy()[:, conv]).all()
                  and np.isfinite(tob.cpu().numpy()[conv]).all())
    # a lone caller: one problem per call through host buffers
    r1 = m.solve_batch(st[:1], cf[:1], want_traj=True, want_mult=True)
    u1 = rng.standard_normal((1, 6))
    for _ in range(10):
        m.solve_batch_jvp(st[:1], cf[:1], r1["traj"], r1["mult"], u1)
    lat = []
    for _ in range(a.lone):
        t0 = time.perf_counter()
        m.solve_batch_jvp(st[:1], cf[:1], r1["traj"], r1["mult"], u1)
        lat.append(1e3 * (time.perf_counter() - t0))
    ms_solve, ms_vjp, ms_jvp = (float(np.median(t)) for t in (t_solve, t_vjp, t_jvp))
    nbytes = jvp_bytes(B, N)
    line = dict(tool="jvp_bench", card=card(), batch=B, N=N, reps=a.reps,
                solve_ms=ms_solve, solve_ms_all=t_solve, vjp_ms=ms_vjp, vjp_ms_all=t_vjp, jvp_ms=ms_jvp, jvp_ms_all=t_jvp,
                jvp_over_solve=ms_jvp / ms_solve, jvp_over_vjp=ms_jvp / ms_vjp,
                jvp_bytes=nbytes, jvp_effective_TBps=nbytes / (ms_jvp * 1e-3) / 1e12,
                converged=int(conv.sum()), jvp_status_ok_on_converged=int((jst[conv] == 0).sum()), finite_on_converged=finite,
                lone_jvp_ms_p50=float(np.percentile(lat, 50)), lone_jvp_ms_p99=float(np.percentile(lat, 99)))
    print(json.dumps(line))
    m.close()


if __name__ == "__main__":
    main()
