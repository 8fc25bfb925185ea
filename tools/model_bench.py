#!/usr/bin/env python
"""Cost of per-problem vehicle models on bench.py's workload (65 536 seeded roadmap problems, degree-3 fits, N = 25).
Arms on device buffers, timed with CUDA events and alternated over --reps repetitions:
    A  solve_batch_warm_device from the default start point, returning the multipliers (the plain entry point)
    B  solve_batch_cost_device with cost8 = the handle's values in every row (same results as A, bit for bit)
    C  solve_batch_model_device with model4 = the handle's values in every row (same results as A, bit for bit)
    D  solve_batch_model_device with seeded random per-problem models: dt uniform in [0.03, 0.1], Lf in [1.5, 4],
       delta_max in [0.2, 0.6], a_max in [0.5, 3]
    vjp / vjp_model  solve_batch_vjp_device and solve_batch_vjp_model_device (broadcast model4, grad_model returned) at
       A's solution
Also the mean and max iterations of every arm and whether B and C matched A bitwise.  Prints one JSON line, with the
card's name and power limit read in the same run.
    python tools/model_bench.py [--batch 65536] [--reps 5] [--seed 0]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip().split(", ")
    return dict(name=q[0], power_limit=q[1] if len(q) > 1 else "unknown")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--seed", type=int, default=0)
    a = ap.parse_args()
    import torch
    import bench
    import udacitympc_b200 as mp
    from udacitympc_b200 import api
    if not torch.cuda.is_available():
        raise SystemExit("model_bench.py needs a CUDA device")
    B, N = a.batch, 25
    dev = torch.device("cuda:0")
    m = mp.MPC(device=0)
    st, cf = bench.make_workload("roadmap", B, mpc=m)
    nv, nm = m.num_vars, m.num_mults
    T = lambda x: torch.from_numpy(np.ascontiguousarray(np.asarray(x, dtype=np.float64).T)).to(dev)
    dst, dcf = T(st), T(cf)
    p = m.params
    c_b = T(np.tile([getattr(p, k) for k in api.PARAM_NAMES], (B, 1)))
    m_c = T(np.tile([getattr(p, k) for k in api.MODEL_NAMES], (B, 1)))
    rng = np.random.default_rng(a.seed)
    lo, hi = np.array([0.03, 1.5, 0.2, 0.5]), np.array([0.1, 4.0, 0.6, 3.0])
    m_d = T(lo + (hi - lo) * rng.uniform(size=(B, 4)))
    E = lambda *s: torch.empty(s, dtype=torch.float64, device=dev)
    I = lambda: torch.empty(B, dtype=torch.int32, device=dev)
    bufs = {arm: dict(out8=E(8, B), traj=E(nv, B), mult=E(nm, B), obj=E(B), status=I(), iters=I()) for arm in "ABCD"}
    g8, gt, go = T(rng.standard_normal((B, 8))), T(rng.standard_normal((B, nv))), torch.from_numpy(rng.standard_normal(B)).to(dev)
    gs, gc, gp, gm, vs = E(6, B), E(4, B), E(8, B), E(4, B), I()
    ts = torch.cuda.Stream()
    torch.cuda.synchronize()   # the inputs were written on the default stream
    torch.cuda.set_stream(ts)
    s = ts.cuda_stream

    def solve(arm):
        o = bufs[arm]
        outs = [o[k].data_ptr() for k in ("out8", "traj", "mult", "obj", "status", "iters")]
        if arm == "A":
            m.solve_batch_warm_device(B, dst.data_ptr(), dcf.data_ptr(), 4, 0, 0, 0.0, *outs, stream=s)
        elif arm == "B":
            m.solve_batch_cost_device(B, dst.data_ptr(), dcf.data_ptr(), 4, c_b.data_ptr(), 0, 0, 0.0, *outs, stream=s)
        else:
            m4 = m_c if arm == "C" else m_d
            m.solve_batch_model_device(B, dst.data_ptr(), dcf.data_ptr(), 4, 0, m4.data_ptr(), 0, 0, 0.0, *outs, stream=s)

    def vjp(model):
        o = bufs["A"]
        args = [dst.data_ptr(), dcf.data_ptr(), 4]
        ins = [o["traj"].data_ptr(), o["mult"].data_ptr(), g8.data_ptr(), gt.data_ptr(), go.data_ptr(), gs.data_ptr(),
               gc.data_ptr(), gp.data_ptr()]
        if model:
            m.solve_batch_vjp_model_device(B, *args, 0, m_c.data_ptr(), *ins, gm.data_ptr(), vs.data_ptr(), s)
        else:
            m.solve_batch_vjp_device(B, *args, *ins, vs.data_ptr(), s)

    def timed(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(ts)
        for _ in range(n):
            fn()
        e1.record(ts)
        e1.synchronize()
        return e0.elapsed_time(e1) / n

    for _ in range(2):   # warm-up: modules, solve graphs, workspace
        for arm in "ABCD":
            solve(arm)
        vjp(False); vjp(True)
    torch.cuda.synchronize()
    t = {k: [] for k in ("A", "B", "C", "D", "vjp", "vjp_model")}
    for _ in range(a.reps):
        for arm in "ABCD":
            t[arm].append(timed(lambda: solve(arm), 3))
        t["vjp"].append(timed(lambda: vjp(False), 10))
        t["vjp_model"].append(timed(lambda: vjp(True), 10))
    torch.cuda.synchronize()
    h = {arm: {k: v.cpu().numpy() for k, v in bufs[arm].items()} for arm in "ABCD"}
    equals_a = lambda arm: all(np.array_equal(h["A"][k], h[arm][k]) for k in h["A"])
    med = {k: float(np.median(v)) for k, v in t.items()}
    conv = lambda arm: float(np.mean((h[arm]["status"] == 0) | (h[arm]["status"] == 1)))
    line = dict(tool="model_bench", card=card(), batch=B, N=N, reps=a.reps,
                ms=med, ms_all=t, solves_per_s={k: B / (med[k] * 1e-3) for k in "ABCD"},
                b_over_a=med["B"] / med["A"], c_over_a=med["C"] / med["A"], d_over_a=med["D"] / med["A"],
                vjp_model_over_vjp=med["vjp_model"] / med["vjp"],
                b_bitwise_equals_a=equals_a("B"), c_bitwise_equals_a=equals_a("C"),
                iters_mean={arm: float(h[arm]["iters"].mean()) for arm in "ABCD"},
                iters_max={arm: int(h[arm]["iters"].max()) for arm in "ABCD"},
                converged={arm: conv(arm) for arm in "ABCD"})
    print(json.dumps(line))
    m.close()


if __name__ == "__main__":
    main()
