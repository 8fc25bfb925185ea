"""Kernel times of the start of a solve: the init kernel and the first rounds of the per-pass sweeps, for one or more
builds of the library (B200MPC_LIB), alternated run by run.

    python tools/first_rounds.py --lib old=/path/libb200mpc.so --lib new=udacitympc_b200/lib/libb200mpc.so --runs 3

Each run is a process of its own (the library is chosen when it is loaded) that solves the bench's roadmap workload
(--batch problems, N = 25) on one stream without the internal batch split, so the kernels of a solve run one after the
other, and records them with torch.profiler (CUDA activity; the trace goes to a temporary directory).  Per build it
prints the median over runs and solves of each of the first launches (init, then factor / forward / step of rounds
1..--rounds) and the span from the start of init to the end of each round; the card's name and power limit go with them.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def child(args):
    sys.path.insert(0, ROOT)
    import torch
    import udacitympc_b200 as mp
    import bench
    m = mp.MPC(device=0)
    m.set_batch_split(1)
    B = args.batch
    st, cf = bench.make_workload("roadmap", B, mpc=m)
    d_st = torch.tensor(np.ascontiguousarray(st.T), device="cuda")
    d_cf = torch.tensor(np.ascontiguousarray(cf.T), device="cuda")
    out8 = torch.empty((8, B), dtype=torch.float64, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    def solve():
        m.solve_batch_device(B, d_st.data_ptr(), d_cf.data_ptr(), cf.shape[1], out8.data_ptr(), stream=stream)

    for _ in range(3):
        solve()
    torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as tmp:
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(args.solves):
                solve()
            torch.cuda.synchronize()
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        ev = json.load(open(path))["traceEvents"]
    kern = sorted((e for e in ev if e.get("cat") == "kernel" and "mpc_" in e.get("name", "")), key=lambda e: e["ts"])
    starts = [i for i, e in enumerate(kern) if "mpc_init_kernel" in e["name"]]
    n = 1 + 3 * args.rounds
    solves = []
    for i in starts:
        seq = kern[i:i + n]
        if len(seq) < n or any("repack" in e["name"] or "coop" in e["name"] for e in seq):
            continue
        t0 = seq[0]["ts"]
        solves.append(dict(dur=[e["dur"] for e in seq],
                           span=[seq[3 * r]["ts"] + seq[3 * r]["dur"] - t0 for r in range(args.rounds + 1)]))
    out = dict(lib=os.environ.get("B200MPC_LIB", "in-tree"), batch=B, solves=solves,
               names=[e["name"].split("<")[0].split("(")[0].split("::")[-1] for e in kern[starts[0]:starts[0] + n]] if starts else [])
    print("RESULT " + json.dumps(out))


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:
        return f"nvidia-smi failed: {e}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", default=[], help="label=path of a libb200mpc.so (repeatable)")
    ap.add_argument("--runs", type=int, default=3, help="processes per build, alternated between the builds")
    ap.add_argument("--solves", type=int, default=5, help="profiled solves per process")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--out", default=None, help="write the per-build summary as JSON here")
    ap.add_argument("--child", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.child:
        return child(args)
    libs = [tuple(s.split("=", 1)) for s in args.lib] or [("in-tree", "")]
    res = {label: [] for label, _ in libs}
    for _ in range(args.runs):
        for label, path in libs:
            env = dict(os.environ)
            if path:
                env["B200MPC_LIB"] = os.path.abspath(path)
            cmd = [sys.executable, os.path.abspath(__file__), "--child", "--solves", str(args.solves), "--rounds",
                   str(args.rounds), "--batch", str(args.batch)]
            r = subprocess.run(cmd, capture_output=True, text=True, env=env, cwd=ROOT)
            line = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")]
            if r.returncode != 0 or not line:
                sys.stderr.write(r.stdout + r.stderr)
                raise SystemExit(f"run of {label} failed")
            res[label].append(json.loads(line[0][7:]))
    gpu = gpu_info()
    summary = dict(gpu=gpu, batch=args.batch, builds={})
    print(f"GPU: {gpu}; {args.batch} problems, N = 25, one stream; medians in microseconds")
    for label, runs in res.items():
        solves = [s for r in runs for s in r["solves"]]
        names = runs[0]["names"]
        dur = np.median(np.array([s["dur"] for s in solves]), axis=0)
        span = np.median(np.array([s["span"] for s in solves]), axis=0)
        summary["builds"][label] = dict(lib=runs[0]["lib"], n_solves=len(solves), kernels=names, kernel_us=dur.tolist(),
                                        init_through_round_us=span.tolist())
        print(f"{label} ({runs[0]['lib']}, {len(solves)} solves)")
        for i, (nm, d) in enumerate(zip(names, dur)):
            rnd = "init" if i == 0 else f"round {(i - 1) // 3 + 1}"
            print(f"  {rnd:8s} {nm:22s} {d:9.1f}")
        print("  init start -> end of " + ", ".join(("init" if r == 0 else f"round {r}") + f" {v:.1f}" for r, v in enumerate(span)))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(summary, f, indent=1)


if __name__ == "__main__":
    main()
