#!/usr/bin/env python
"""Cost of per-problem cost parameters on bench.py's workload (65 536 seeded roadmap problems, degree-3 fits, N = 25).
Arms on device buffers, timed with CUDA events and alternated over --reps repetitions:
    A  solve_batch_warm_device from the default start point, returning the multipliers (the plain entry point)
    B  solve_batch_cost_device with cost8 = the handle's values in every row (same results as A, bit for bit)
    C  solve_batch_cost_device with random per-problem costs: ref_v uniform in [10, 60], weights log-uniform in
       [0.1, 100], seeded
    vjp / vjp_cost  solve_batch_vjp_device and solve_batch_vjp_cost_device (broadcast costs) at A's solution
Also the iterations of A and C and whether B matched A bitwise.  Prints one JSON line, with the card's name and power
limit read in the same run.
    python tools/cost_bench.py [--batch 65536] [--reps 5] [--seed 0]"""
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
        raise SystemExit("cost_bench.py needs a CUDA device")
    B, N = a.batch, 25
    dev = torch.device("cuda:0")
    m = mp.MPC(device=0)
    st, cf = bench.make_workload("roadmap", B, mpc=m)
    nv, nm = m.num_vars, m.num_mults
    T = lambda x: torch.from_numpy(np.ascontiguousarray(np.asarray(x, dtype=np.float64).T)).to(dev)
    dst, dcf = T(st), T(cf)
    p = m.params
    c_b = T(np.tile([getattr(p, k) for k in api.PARAM_NAMES], (B, 1)))
    rng = np.random.default_rng(a.seed)
    c_c = T(np.concatenate([rng.uniform(10.0, 60.0, (B, 1)), 10.0 ** rng.uniform(-1.0, 2.0, (B, 7))], axis=1))
    E = lambda *s: torch.empty(s, dtype=torch.float64, device=dev)
    I = lambda: torch.empty(B, dtype=torch.int32, device=dev)
    bufs = {arm: dict(out8=E(8, B), traj=E(nv, B), mult=E(nm, B), obj=E(B), status=I(), iters=I()) for arm in "ABC"}
    g8, gt, go = T(rng.standard_normal((B, 8))), T(rng.standard_normal((B, nv))), torch.from_numpy(rng.standard_normal(B)).to(dev)
    gs, gc, gp, vs = E(6, B), E(4, B), E(8, B), I()
    ts = torch.cuda.Stream()
    torch.cuda.synchronize()   # the inputs were written on the default stream
    torch.cuda.set_stream(ts)
    s = ts.cuda_stream

    def solve(arm):
        o = bufs[arm]
        outs = [o[k].data_ptr() for k in ("out8", "traj", "mult", "obj", "status", "iters")]
        if arm == "A":
            m.solve_batch_warm_device(B, dst.data_ptr(), dcf.data_ptr(), 4, 0, 0, 0.0, *outs, stream=s)
        else:
            c8 = c_b if arm == "B" else c_c
            m.solve_batch_cost_device(B, dst.data_ptr(), dcf.data_ptr(), 4, c8.data_ptr(), 0, 0, 0.0, *outs, stream=s)

    def vjp(cost):
        o = bufs["A"]
        args = [dst.data_ptr(), dcf.data_ptr(), 4]
        tail = [o["traj"].data_ptr(), o["mult"].data_ptr(), g8.data_ptr(), gt.data_ptr(), go.data_ptr(), gs.data_ptr(),
                gc.data_ptr(), gp.data_ptr(), vs.data_ptr(), s]
        if cost:
            m.solve_batch_vjp_cost_device(B, *args, c_b.data_ptr(), *tail)
        else:
            m.solve_batch_vjp_device(B, *args, *tail)

    def timed(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(ts)
        for _ in range(n):
            fn()
        e1.record(ts)
        e1.synchronize()
        return e0.elapsed_time(e1) / n

    for _ in range(2):   # warm-up: modules, solve graphs, workspace
        for arm in "ABC":
            solve(arm)
        vjp(False); vjp(True)
    torch.cuda.synchronize()
    t = {k: [] for k in ("A", "B", "C", "vjp", "vjp_cost")}
    for _ in range(a.reps):
        for arm in "ABC":
            t[arm].append(timed(lambda: solve(arm), 3))
        t["vjp"].append(timed(lambda: vjp(False), 10))
        t["vjp_cost"].append(timed(lambda: vjp(True), 10))
    torch.cuda.synchronize()
    h = {arm: {k: v.cpu().numpy() for k, v in bufs[arm].items()} for arm in "ABC"}
    b_equals_a = all(np.array_equal(h["A"][k], h["B"][k]) for k in h["A"])
    med = {k: float(np.median(v)) for k, v in t.items()}
    conv = lambda arm: float(np.mean((h[arm]["status"] == 0) | (h[arm]["status"] == 1)))
    line = dict(tool="cost_bench", card=card(), batch=B, N=N, reps=a.reps,
                ms=med, ms_all=t, solves_per_s={k: B / (med[k] * 1e-3) for k in "ABC"},
                b_over_a=med["B"] / med["A"], c_over_a=med["C"] / med["A"], vjp_cost_over_vjp=med["vjp_cost"] / med["vjp"],
                b_bitwise_equals_a=b_equals_a,
                iters_mean={arm: float(h[arm]["iters"].mean()) for arm in "AC"},
                iters_max={arm: int(h[arm]["iters"].max()) for arm in "AC"},
                converged={arm: conv(arm) for arm in "AC"})
    print(json.dumps(line))
    m.close()


if __name__ == "__main__":
    main()
