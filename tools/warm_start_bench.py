#!/usr/bin/env python
"""Warm-started receding horizon on bench.py's workload (65 536 seeded roadmap problems, degree-3 fits): K steps, each
starting from the previous step's out8 as closed_loop does, the reference polynomial held fixed.  Three throughput arms,
run alternated in one process:
    cold        solve_batch_device every step (the reference's cold start)
    warm        solve_batch_warm_device from the previous step's traj / mult, shifted by shift_solution on the device
    closed_loop closed_loop_batch with set_warm_start (the solution stays in the workspace; no batch compaction)
and the latency of a lone caller (one problem per call, host buffers): cold vs warm from the shifted previous solution.
Prints one JSON line, with the card's name and power limit read in the same run.
    python tools/warm_start_bench.py [--batch 65536] [--steps 10] [--reps 3] [--lone 200]"""
import argparse
import json
import os
import subprocess
import sys
import time

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
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--lone", type=int, default=200)
    a = ap.parse_args()
    import torch
    import bench
    import udacitympc_b200 as mp
    B, K, N = a.batch, a.steps, 25
    dev = torch.device("cuda:0")
    m = mp.MPC(device=0)
    mcl = mp.MPC(device=0)
    mcl.set_warm_start(True, 1e-4)
    st, cf = bench.make_workload("roadmap", B, mpc=m)
    nv, nm = m.num_vars, m.num_mults
    T = lambda x: torch.from_numpy(np.ascontiguousarray(x.T)).to(dev)
    st0, dcf = T(st), T(cf)
    # fixed buffers: a solve graph is cached per set of buffer addresses (b200mpc's graph key)
    state = torch.empty_like(st0)
    out8 = torch.empty((8, B), dtype=torch.float64, device=dev)
    iters = torch.empty(B, dtype=torch.int32, device=dev)
    traj = torch.empty((nv, B), dtype=torch.float64, device=dev); mult = torch.empty((nm, B), dtype=torch.float64, device=dev)
    x0 = torch.empty_like(traj); m0 = torch.empty_like(mult)
    ts = torch.cuda.Stream()   # the solves and the torch work that feeds them on one stream
    torch.cuda.set_stream(ts)
    s = ts.cuda_stream

    def cold():
        state.copy_(st0); o, it = [], []
        for _ in range(K):
            m.solve_batch_device(B, state.data_ptr(), dcf.data_ptr(), 4, out8.data_ptr(), d_iters=iters.data_ptr(), stream=s)
            state.copy_(out8[:6]); o.append(out8.clone()); it.append(iters.clone())
        return o, it

    def warm():
        state.copy_(st0); o, it = [], []
        for k in range(K):
            m.solve_batch_warm_device(B, state.data_ptr(), dcf.data_ptr(), 4, x0.data_ptr() if k else 0, m0.data_ptr() if k else 0,
                                      1e-4, out8.data_ptr(), traj.data_ptr(), mult.data_ptr(), d_iters=iters.data_ptr(), stream=s)
            xs, ms = mp.shift_solution(traj, mult, N, field_major=True)
            x0.copy_(xs); m0.copy_(ms); state.copy_(out8[:6]); o.append(out8.clone()); it.append(iters.clone())
        return o, it

    def closed_loop():
        r = mcl.closed_loop(st, cf, K)
        return [torch.from_numpy(np.ascontiguousarray(r["hist8"][k].T)) for k in range(K)], [torch.from_numpy(r["iters"][k]) for k in range(K)]

    arms = dict(cold=cold, warm=warm, closed_loop=closed_loop)
    times = {k: [] for k in arms}
    res = {}
    for rep in range(a.reps + 1):   # rep 0: warm-up (graph capture, module load)
        for name, f in arms.items():
            torch.cuda.synchronize(); t = time.perf_counter()
            o, it = f()
            torch.cuda.synchronize(); dt = time.perf_counter() - t
            if rep:
                times[name].append(dt)
            res[name] = ([x.cpu().numpy() for x in o], np.stack([x.cpu().numpy() for x in it]))
    out = dict(tool="warm_start_bench", card=card(), batch=B, steps=K, N=N, reps=a.reps)
    for name in arms:
        its = res[name][1][1:]   # steps 2..K: step 1 is a cold start in every arm
        out[name] = dict(solves_per_s=B * K / float(np.mean(times[name])), time_s=[round(x, 4) for x in times[name]],
                         iters_mean=float(its.mean()), iters_max=int(its.max()))
    ref = np.stack(res["cold"][0])
    for n in ("warm", "closed_loop"):   # per problem, over the K steps: a trajectory that leaves the road can diverge
        d = np.abs(np.stack(res[n][0]) - ref).max(axis=(0, 1))
        out[f"dout8_{n}"] = dict(max=float(d.max()), p99=float(np.percentile(d, 99)), over_1e_6=int((d > 1e-6).sum()))
    # lone caller: problem i's next step (state = its out8[:6]), cold vs warm from its shifted solution, alternated
    n = min(a.lone, B)
    first = m.solve_batch(st[:n], cf[:n], want_traj=True, want_mult=True)
    xs, ms = mp.shift_solution(first["traj"], first["mult"], N)
    nxt = np.ascontiguousarray(first["out8"][:, :6])
    lat = dict(cold=[], warm=[])
    for rep in range(2):
        for i in range(n):
            for kind in ("cold", "warm"):
                kw = dict(x_init=xs[i:i + 1], mult_init=ms[i:i + 1]) if kind == "warm" else {}
                t = time.perf_counter()
                m.solve_batch(nxt[i:i + 1], cf[i:i + 1], **kw)
                if rep:
                    lat[kind].append(time.perf_counter() - t)
    for kind, v in lat.items():
        out[f"lone_{kind}_ms"] = dict(p50=float(np.percentile(v, 50) * 1e3), p99=float(np.percentile(v, 99) * 1e3))
    print(json.dumps(out))
    m.close(); mcl.close()


if __name__ == "__main__":
    main()
