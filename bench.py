#!/usr/bin/env python
"""bench.py -- MPC solves/sec (BASELINE.json metric) for the B200-native batched MPC solver.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch B] [--workload roadmap|line]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic input: B = 65 536 independent MPC::Solve problems
(N=25 horizon).  Default workload = BASELINE.json configs[3]: a degree-3 reference fitted (on the GPU, K4) to
roadmap.csv segments, ONE batch per step sharded by problem index over the GPUs ("scaling": "strong"; rank r of N
solves problems [r*B/N, (r+1)*B/N), udacitympc_b200/sharding.py).  There is no data-path collective;
torch.distributed (NCCL) is used only for the barrier and the max-over-ranks of the device time.  --scaling weak
gives every GPU its own B problems per step instead.

value        whole-job solves/s with inputs already resident in HBM (device-pointer C-ABI call, CUDA events; the timed
             region is exactly K steps)
e2e          the same through the host-buffer C-ABI call the reference's MPC::Solve would bind: pinned host buffers,
             H2D + D2H inside the timed region (K steps)
lone_caller  one handle, one stream, one call at a time (the figures above overlap consecutive steps on several handles)
one_process_multi_gpu (N > 1)  b200mpc_solve_batch_multi on the whole batch from rank 0: every GPU's shard queued from one host thread, host
             gather, per-call latency percentiles
weak_scaling (N > 1)  the weak-scaling figure next to the strong one

--dump-outputs DIR writes what the last timed step returned to its caller (out8 (8, B), obj, status, iters of the whole
batch, as float64 .npy files; a fixed sample of problems with its index.npy when that would exceed 64 MB).  The inputs
are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import multiprocessing as mp_
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "mpc_solves_per_sec"
UNIT = "solves/s"
HORIZON = 25


def f_iter(N):
    """Algorithmic FLOP per interior-point iteration per problem (SURVEY 8d): (N-1)(F_ric + F_eval) + F_vec N."""
    return (N - 1) * (2421 + 150) + 20 * N


def profiled_traffic_bytes():
    """DRAM bytes (read + write) of all solver kernels of ONE step, from the committed ncu launch list of this same
    command (profiles/r1_compact_launches_time_dram.csv: one init ... next init).  None if the file is missing."""
    import csv
    path = os.path.join(ROOT, "profiles", "r1_compact_launches_time_dram.csv")
    try:
        rows = [r for r in csv.reader(open(path)) if len(r) > 5]
        hdr = rows[0]
        ik, iv, im, iu, iid = (hdr.index(c) for c in ("Kernel Name", "Metric Value", "Metric Name", "Metric Unit", "ID"))
        per = {}
        for r in rows[1:]:
            if "dram__bytes" not in r[im]:
                continue
            scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(r[iu], 1.0)
            d = per.setdefault(int(r[iid]), [r[ik], 0.0])
            d[1] += float(r[iv].replace(",", "")) * scale
        seq = [per[k] for k in sorted(per)]
        starts = [i for i, (k, _) in enumerate(seq) if "mpc_init_kernel" in k]
        if len(starts) < 2:
            return None
        return float(sum(b for k, b in seq[starts[0]:starts[1]] if "mpc_" in k))
    except Exception:
        return None


def profiled_counters():
    """Per-step counters that come from committed ncu captures of this same command (one GPU, 65 536 problems per step):
    profiles/r2_counters.json (written by tools/ncu_counters.py from the launch list) when present, else the round-1
    launch list (DRAM bytes only)."""
    path = os.path.join(ROOT, "profiles", "r2_counters.json")
    try:
        d = json.load(open(path))
        if d.get("dram_bytes_per_step"):
            return d
    except Exception:
        pass
    t = profiled_traffic_bytes()
    return dict(dram_bytes_per_step=t,
                traffic_unit="bytes of DRAM read+write of all solver kernels of one 65 536-problem step (ncu, profiles/r1_compact_launches_time_dram.csv)")


def make_workload(kind, B, seed_shift=0, mpc=None):
    """Returns (states (B,6), coeffs (B,ncoef)).  Degree-3 coefficients come from the GPU polyfit when a handle is
    given (that is the product path); the CPU-only reference arm uses numpy's QR for its own inputs."""
    from udacitympc_b200 import synth
    rng = synth.MT19937_64(synth.SEED + 1000 * seed_shift)
    if kind == "line":
        return synth.line_problems(B, rng)
    xs, ys = synth.roadmap_windows(B, rng)
    if mpc is not None:
        import udacitympc_b200 as m
        fit = m.polyfit_batch(xs, ys, 3, mpc=mpc)
    else:
        V = np.stack([xs ** i for i in range(4)], axis=2)
        fit = np.stack([np.linalg.lstsq(V[b], ys[b], rcond=None)[0] for b in range(B)])
    st = synth.roadmap_problems(B, fit, synth.MT19937_64(synth.SEED + 1 + 1000 * seed_shift))
    return st, np.ascontiguousarray(fit)


# ------------------------------------------------------------------------------------------------
# CPU reference arm: the reference's own Ipopt 3.12.7 + MUMPS binaries (oracle/_ref), one process per host core.
def _cpu_worker(args):
    kind, states, coeffs = args
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_bindings as ob
    t0 = time.perf_counter()
    its = 0
    for b in range(len(states)):
        r = ob.ref_solve(states[b], coeffs[b]) if kind == "reference" else ob.port_solve(states[b], coeffs[b])
        its += r["iters"]
    return time.perf_counter() - t0, its


def cpu_reference_rate(states, coeffs, per_core, cores=None):
    """Times the reference CPU implementation on a bounded sample: `per_core` solves on each of `cores` processes."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_bindings as ob
    kind = "reference" if ob.ref_available() else "port"
    cores = cores or os.cpu_count() or 1
    n = min(len(states), cores * per_core)
    per = max(1, n // cores)
    chunks = [(kind, states[i * per:(i + 1) * per], coeffs[i * per:(i + 1) * per]) for i in range(cores)]
    chunks = [c for c in chunks if len(c[1])]
    ctx = mp_.get_context("fork")
    t0 = time.perf_counter()
    with ctx.Pool(len(chunks)) as pool:
        res = pool.map(_cpu_worker, chunks)
    wall = time.perf_counter() - t0
    solved = sum(len(c[1]) for c in chunks)
    busy = max(r[0] for r in res)
    iters = sum(r[1] for r in res)
    return dict(value=solved / busy, unit=UNIT, cores=len(chunks), kind=kind, solved=solved,
                sample=f"first {solved} problems of the workload, {per} per process ({busy:.2f} s of CPU work on the slowest), one process per host core "
                       f"(Ipopt 3.12.7 + MUMPS 4.10.0 reference binaries, hand-derived derivatives standing in for CppAD)"
                if kind == "reference" else f"first {solved} problems, C port of the reference algorithm",
                wall_s=wall, mean_iters=iters / max(1, solved))


def run_reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path (oracle/_ref = its Ipopt 3.12.7 + MUMPS
    binaries; the C port when they are absent) on every host core, on a bounded sample of the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_bindings as ob
    ob.ref_available() and ob.ref()   # dlopen oracle/_ref/libmpc_ref.so in THIS process too (the solves run in forked workers)
    states, coeffs = make_workload(args.workload, min(args.batch, 8192))
    cores = os.cpu_count() or 1
    per_core = args.ref_per_core   # solves per host core per step: >= 1 s of CPU work per core and step
    times = []
    rate = None
    for i in range(args.warmup + args.steps):
        r = cpu_reference_rate(states, coeffs, per_core, cores)
        if i >= args.warmup:
            times.append(r["solved"] / r["value"])
            rate = r
    solved_per_step = rate["solved"]
    ms = 1e3 * float(np.mean(times))
    value = solved_per_step / (ms * 1e-3)
    line = dict(metric=METRIC, value=value, unit=UNIT, impl="reference", n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=ms, higher_is_better=True, scaling=args.scaling, vs_baseline=None, dtype="f64",
                data="synthetic", config=config_dict(args),
                solved_per_step=solved_per_step,
                note=f"each step of this arm solves a bounded sample of the workload ({solved_per_step} problems = {per_core} per host "
                     f"core), not all {args.batch}; value = solved problems per second of wall time of the slowest worker",
                cpu_baseline=dict(value=value, unit=UNIT, cores=rate["cores"], kind=rate["kind"], sample=rate["sample"]),
                e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    emit(line)


def config_dict(args):
    """The workload both arms are measured on (identical in the two JSON lines)."""
    return dict(workload=("BASELINE configs[3]: batched MPC, 65 536 problems per step, degree-3 reference fitted to roadmap.csv segments, "
                          "one batch sharded by index over the GPUs" if args.workload == "roadmap" else
                          "BASELINE configs[2]: batched mpc_to_line, degree-1 reference y=-1"),
                horizon_N=HORIZON, dt=0.05, problems_per_step=args.batch,
                sharding="contiguous index ranges per GPU (rank r solves [r*B/N, (r+1)*B/N)), no collective, results gathered by the host",
                l2="per-step working set (solver workspace, 17.9 KB per problem in flight) >> 126 MB L2; the inputs cycle over "
                   "4 distinct 65 536-problem batches")


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,utilization.gpu")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                busy = float(r[7]) > 50.0 if len(r) > 7 else True
                if busy:   # median under load: idle samples (workload generation, CPU legs) would only dilute it
                    sm.append(float(r[0]))
                mx.append(float(r[1]))
                for nme, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                pass
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=float(max(mx)) if mx else None,
                    reasons=sorted(reasons), samples=len(self.rows), samples_under_load=len(sm))


DUMP_MAX_BYTES = 64 * 10 ** 6


def dump_outputs(path, outs):
    """Writes the per-problem result arrays `outs` (problem index on the last axis) to path/<name>.npy as float64.  When
    they would take more than DUMP_MAX_BYTES, a fixed seeded sample of problems is written instead, with its indices
    (index.npy), so that the same arguments always select the same problems."""
    n = next(iter(outs.values())).shape[-1]
    per_problem = 8 * (sum(int(np.prod(a.shape[:-1])) for a in outs.values()) + 1)
    budget = DUMP_MAX_BYTES - 4096   # room for the .npy headers
    os.makedirs(path, exist_ok=True)
    if n * per_problem > budget:
        idx = np.sort(np.random.default_rng(0).choice(n, budget // per_problem, replace=False))
        outs = {k: a[..., idx] for k, a in outs.items()}
        np.save(os.path.join(path, "index.npy"), idx.astype(np.float64))
    for k, a in outs.items():
        np.save(os.path.join(path, f"{k}.npy"), np.ascontiguousarray(a, dtype=np.float64))


def auto_streams(per_gpu_batch):
    """Solver handles / streams whose consecutive steps overlap: 6 at 65 536 problems per GPU and step, more for the
    smaller per-GPU shards of a strong-scaled batch (about 6 x 65 536 problems in flight per GPU), at most 16."""
    return int(min(16, max(6, round(6 * 65536 / max(1, per_gpu_batch)))))


def run_ours(args):
    # one hardware work queue per overlapped stream (the default of 8 makes 12-16 streams share queues: kernels of one
    # stream then wait behind another stream's); read by the CUDA runtime when the context is created
    os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
    import ctypes
    import math
    from concurrent.futures import ThreadPoolExecutor

    import torch
    import torch.distributed as dist
    import udacitympc_b200 as mpcmod
    from udacitympc_b200 import api as mpcapi
    from udacitympc_b200.sharding import max_over_ranks, shard_range, throughput

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU path (use --impl reference for the CPU arm)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"   # keep NCCL's version banner off stdout: rank 0 prints exactly one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    # the ranks that sit out the one-process leg wait on the host (gloo), not inside an NCCL kernel on their GPU
    cpu_group = dist.new_group(backend="gloo") if world > 1 else None
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    B, K, W = args.batch, args.steps, args.warmup
    strong = args.scaling == "strong"
    # strong (default, BASELINE configs[3]): ONE B-problem batch per step, rank r solves its index range of it;
    # weak: every rank solves all B problems of its own copy
    lo, hi = shard_range(B, world, rank) if strong else (0, B)
    Bl = hi - lo
    total_per_step = B if strong else B * world

    S = args.streams if args.streams > 0 else auto_streams(Bl)
    # concurrency comes either from the caller (S overlapped handles, no internal split) or from the library's
    # internal batch split (one handle)
    split = args.split if args.split > 0 else (1 if S > 1 else 4)
    mpcs = [mpcmod.MPC(device=local) for _ in range(S)]
    for m in mpcs:
        m.set_solver_mode({"perpass": 0, "fused": 1}[args.mode], args.rounds, -1)
        m.set_batch_split(split)
        if S > 1 and args.handover >= 0:
            m.set_handover(args.handover, 14)   # overlapped calls: a later hand-over to the cooperative kernel (b200mpc_set_handover)
    # --pipeline D: the device-timed region issues its S overlapped streams to ONE handle in pipelined mode (bulk in one
    # full-size workspace, tails in D small contexts) instead of S handles with a full-size workspace each
    dev_handles = mpcs
    if args.pipeline > 0:
        mpcs[0].set_pipeline(args.pipeline, args.pipeline_slots if args.pipeline_slots > 0 else max(1024, Bl // 16))
        dev_handles = [mpcs[0]] * S
    mpc = mpcs[0]
    # Four distinct B-problem input sets, cycled step by step (every rank generates the same sets and keeps its index
    # range); about half of such sets contain a 30-50 iteration straggler (DESIGN.md 4), so cycling several makes the
    # figure representative of the workload.
    nsets = args.input_sets
    sets = [make_workload(args.workload, B, seed_shift=s, mpc=mpc) for s in range(nsets)]
    ncoef = sets[0][1].shape[1]

    def device_inputs(a, b):   # field-major device copies of problems [a, b) of every set
        return [(torch.from_numpy(np.ascontiguousarray(st[a:b].T)).to(dev), torch.from_numpy(np.ascontiguousarray(cf[a:b].T)).to(dev))
                for st, cf in sets]

    def device_outputs(n, count):
        return [dict(out8=torch.empty((8, n), dtype=torch.float64, device=dev), obj=torch.empty(n, dtype=torch.float64, device=dev),
                     status=torch.empty(n, dtype=torch.int32, device=dev), iters=torch.empty(n, dtype=torch.int32, device=dev))
                for _ in range(count)]

    d_in = device_inputs(lo, hi)
    d_out = device_outputs(Bl, S)
    # real (non-default) streams: kernels and timing events share them.  With S > 1 consecutive steps alternate
    # between S solver handles / streams so that the thin tail of one batch (few problems still iterating)
    # overlaps the bulk of the next.
    streams = [torch.cuda.Stream(device=dev) for _ in range(S)]
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_device_region(handles, strs, n, ins, outs, steps):
        """`steps` solves of n problems, step i on handle / stream i % len(handles); device time in ms (CUDA events on
        the launching streams: e0 before the first launch, e1 after every stream has drained into stream 0)."""
        ns = len(handles)

        def one(i):
            st, cf = ins[i % nsets]
            o = outs[i % ns]
            handles[i % ns].solve_batch_device(n, st.data_ptr(), cf.data_ptr(), ncoef, o["out8"].data_ptr(), 0, o["obj"].data_ptr(),
                                               o["status"].data_ptr(), o["iters"].data_ptr(), strs[i % ns].cuda_stream)

        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(strs[0])
        for s_ in strs[1:]:
            s_.wait_event(e0)
        for i in range(steps):
            one(i)
        for s_ in strs[1:]:
            ev = torch.cuda.Event()
            ev.record(s_)
            strs[0].wait_event(ev)
        e1.record(strs[0])
        return e0, e1

    def agreed(ms):   # the same number on every rank (max), so that every rank runs the same number of steps
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        return max_over_ranks(dist, t, world)

    fp64_peak = mpc.fp64_peak_tflops()
    # warm-up: at least W steps, and every (solver handle, input set) pair once -- each pair is its own CUDA graph,
    # captured and instantiated at its first use
    wsteps = max(W, S * nsets // math.gcd(S, nsets))
    timed_device_region(dev_handles, streams, Bl, d_in, d_out, wsteps)
    barrier()
    launches0 = sum(m.launch_count() for m in mpcs)
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    e0, e1 = timed_device_region(dev_handles, streams, Bl, d_in, d_out, K)
    barrier()
    ms_total, per_rank_total = agreed(e0.elapsed_time(e1))
    launches = sum(m.launch_count() for m in mpcs) - launches0
    per_rank_ms = [x / K for x in per_rank_total]
    value = throughput(total_per_step, K, ms_total)
    if args.dump_outputs:   # step K - 1 wrote the output set of its handle, which no later leg touches
        last = {k: v.cpu().numpy() for k, v in d_out[(K - 1) % len(dev_handles)].items()}
        if world > 1:   # rank 0 writes the whole batch (strong) or its own copy of it (weak)
            shards = [None] * world if rank == 0 else None
            dist.gather_object(last, shards, dst=0, group=cpu_group)
            if rank == 0 and strong:
                last = {k: np.concatenate([s[k] for s in shards], axis=-1) for k in last}
        if rank == 0:
            dump_outputs(args.dump_outputs, last)

    # ---- one caller, one call at a time: 1 handle (library defaults: the call is cut into 4 concurrent sub-batches
    # inside), 1 stream; every solve bracketed by CUDA events inside the C ABI (b200mpc_set_timing)
    lone = mpcmod.MPC(device=local)
    lone.set_solver_mode({"perpass": 0, "fused": 1}[args.mode], args.rounds, -1)
    lone.set_timing(True)
    lone_out = device_outputs(Bl, 1)
    n_lone = max(K, 2 * nsets)
    timed_device_region([lone], streams[:1], Bl, d_in, lone_out, nsets)   # graphs
    barrier()
    lone.kernel_time_ms(reset=True)
    e0, e1 = timed_device_region([lone], streams[:1], Bl, d_in, lone_out, n_lone)
    barrier()
    lone_ms, _ = agreed(e0.elapsed_time(e1))
    lone_kern_ms, lone_kern_n = lone.kernel_time_ms(reset=True)
    lone_value = throughput(total_per_step, n_lone, lone_ms)
    # mean iterations / solved fraction of this rank's share of every input set
    iters_sum, ok_sum = 0.0, 0.0
    for s in range(nsets):
        timed_device_region([lone], streams[:1], Bl, d_in[s:] + d_in[:s], lone_out, 1)
        torch.cuda.synchronize()
        iters_sum += float(lone_out[0]["iters"].double().sum().item())
        ok_sum += float((lone_out[0]["status"] == 0).double().sum().item())
    tt = torch.tensor([iters_sum, ok_sum, float(Bl * nsets)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.SUM)
    mean_it, solved_fraction = float(tt[0] / tt[2]), float(tt[1] / tt[2])
    lone.set_timing(False)

    # ---- e2e: host buffers (pinned), H2D + D2H inside the timed region, through the host-buffer C-ABI call;
    # T host threads, one solver handle each (the call blocks until its results are in the caller's buffers)
    pin = [(torch.from_numpy(np.ascontiguousarray(st[lo:hi])).pin_memory(), torch.from_numpy(np.ascontiguousarray(cf[lo:hi])).pin_memory())
           for st, cf in sets]
    lib = mpcmod.load_library()
    dp, ip = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int)

    def host_outputs(n):
        return dict(out8=torch.empty((n, 8), dtype=torch.float64).pin_memory(), obj=torch.empty(n, dtype=torch.float64).pin_memory(),
                    status=torch.empty(n, dtype=torch.int32).pin_memory(), iters=torch.empty(n, dtype=torch.int32).pin_memory())

    hout = [host_outputs(Bl) for _ in range(S)]

    if args.pipeline > 0:
        torch.cuda.synchronize()
        mpcs[0].set_pipeline(0, 0)   # the host-buffer calls below block: one handle per host thread, as without --pipeline

    def host_step(i, k, handle=None, out=None, wait=True):
        st, cf = pin[i % nsets]
        o = out or hout[k]
        fn = lib.b200mpc_solve_batch if wait else lib.b200mpc_solve_batch_async
        rc = fn((handle or mpcs[k]).handle, Bl, ctypes.cast(st.data_ptr(), dp), ctypes.cast(cf.data_ptr(), dp), ncoef,
                ctypes.cast(o["out8"].data_ptr(), dp), None, ctypes.cast(o["obj"].data_ptr(), dp),
                ctypes.cast(o["status"].data_ptr(), ip), ctypes.cast(o["iters"].data_ptr(), ip))
        if rc:
            raise RuntimeError(lib.b200mpc_last_error().decode())

    # host threads of the end-to-end leg (one solver handle each): one per handle, but not more than the rank's share
    # of the host cores (never fewer than 3)
    T = args.e2e_threads if args.e2e_threads > 0 else min(S, max(3, (os.cpu_count() or 6) // world))
    T = max(1, min(S, T))

    # host thread k drives the handles k, k + T, k + 2T, ... (one pinned output set each): it queues a step on each of
    # them with the asynchronous host-buffer call and waits for a handle's previous step (b200mpc_wait: its results are
    # then in the caller's buffers) just before giving it the next one, so S calls are in flight per GPU whatever the
    # number of host cores.  With T = S this is one blocking call per thread, as the reference's MPC::Solve would be used.
    def worker(k, n):
        mine = list(range(k, S, T))
        busy = {h: False for h in mine}
        j = 0
        for i in range(k, n, T):
            h = mine[j % len(mine)]
            j += 1
            if busy[h]:
                mpcs[h].wait()
            host_step(i, h, wait=False)
            busy[h] = True
        for h in mine:
            if busy[h]:
                mpcs[h].wait()

    for i in range(max(3, S)):   # every handle of the leg allocates its staging buffers and captures its graph here
        host_step(i, i % S)
    barrier()
    n_e2e = K
    with ThreadPoolExecutor(T) as ex:
        t0 = time.perf_counter()
        list(ex.map(lambda k: worker(k, n_e2e), range(T)))
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
    e2e_max_s, _ = agreed(e2e_s)
    e2e_value = total_per_step * n_e2e / e2e_max_s
    # unloaded latency of one host-buffer call at a time (the lone handle: library defaults)
    lat = []
    for i in range(3):
        host_step(i, 0, lone, hout[0])
    for i in range(args.latency_reps):
        a = time.perf_counter()
        host_step(i, 0, lone, hout[0])
        lat.append(time.perf_counter() - a)
    p99, _ = agreed(float(np.percentile(lat, 99)))
    p50, _ = agreed(float(np.percentile(lat, 50)))
    clocks = sampler.stop()
    cmhz, per_rank_mhz = agreed(clocks.get("sm_mhz") or 0.0)

    # ---- one process, every GPU's shard queued from one host thread, host gather: b200mpc_solve_batch_multi on the WHOLE batch (rank 0
    # only, the other ranks wait; SURVEY 8e "results gathered by the host")
    multi = None
    barrier()
    if world > 1 and rank == 0 and strong and torch.cuda.device_count() >= world and not args.no_multi_leg:
        hs = [mpcmod.MPC(device=d) for d in range(world)]
        try:
            full = [(torch.from_numpy(st).pin_memory(), torch.from_numpy(cf).pin_memory()) for st, cf in sets]
            fo = host_outputs(B)
            harr = (ctypes.c_void_p * world)(*[h.handle for h in hs])

            def multi_step(i):
                st, cf = full[i % nsets]
                rc = lib.b200mpc_solve_batch_multi(harr, world, B, ctypes.cast(st.data_ptr(), dp), ctypes.cast(cf.data_ptr(), dp), ncoef,
                                                   ctypes.cast(fo["out8"].data_ptr(), dp), None, ctypes.cast(fo["obj"].data_ptr(), dp),
                                                   ctypes.cast(fo["status"].data_ptr(), ip), ctypes.cast(fo["iters"].data_ptr(), ip))
                if rc:
                    raise RuntimeError(lib.b200mpc_last_error().decode())

            for i in range(nsets + 1):
                multi_step(i)
            ml = []
            for i in range(args.latency_reps):
                a = time.perf_counter()
                multi_step(i)
                ml.append(time.perf_counter() - a)
            multi = dict(entry="b200mpc_solve_batch_multi", handles=world, problems_per_call=B, calls=len(ml), host_buffers="pinned",
                         value=B / float(np.mean(ml)), unit=UNIT, p50_batch_latency_ms=1e3 * float(np.percentile(ml, 50)),
                         p99_batch_latency_ms=1e3 * float(np.percentile(ml, 99)), solved_fraction=float((fo["status"] == 0).double().mean()))
        finally:
            for h in hs:
                h.close()
    if world > 1:
        dist.barrier(group=cpu_group)
    barrier()

    # ---- weak-scaling figure next to the strong one (N > 1): every rank solves a whole B-problem batch per step
    weak = None
    if world > 1 and strong and not args.no_weak_leg:
        Sw = min(S, 6)
        w_in = device_inputs(0, B)
        w_out = device_outputs(B, Sw)
        timed_device_region(mpcs[:Sw], streams[:Sw], B, w_in, w_out, max(3, Sw * nsets // math.gcd(Sw, nsets)))
        barrier()
        e0, e1 = timed_device_region(mpcs[:Sw], streams[:Sw], B, w_in, w_out, max(K, 20))
        barrier()
        wms, _ = agreed(e0.elapsed_time(e1))
        weak = dict(value=throughput(B * world, max(K, 20), wms), unit=UNIT, problems_per_gpu_per_step=B, steps=max(K, 20), streams=Sw)

    if rank == 0:
        flop_per_step = f_iter(HORIZON) * mean_it * total_per_step
        # device time of the solver kernels per step, read both ways: (a) with S overlapped streams the per-step share of
        # the timed region (the intervals of consecutive steps overlap); (b) one stream, one call at a time: the
        # first-to-last-kernel interval of each solve (CUDA events inside the C ABI)
        avg_kernel_ms = ms_total / K
        lone_kernel_ms = lone_kern_ms / max(1, lone_kern_n)
        achieved = flop_per_step / (avg_kernel_ms * 1e-3) / 1e12 / world      # per GPU
        lone_achieved = f_iter(HORIZON) * mean_it * Bl / (lone_kernel_ms * 1e-3) / 1e12
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        prof = profiled_counters()
        traffic = prof.get("dram_bytes_per_step")
        line = dict(
            metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=K, warmup=W, ms_per_step=ms_total / K,
            higher_is_better=True, scaling=args.scaling, vs_baseline=None, dtype="f64", data="synthetic",
            config=config_dict(args),
            timed=dict(passes=K, seconds=ms_total * 1e-3, problems_per_gpu_per_step=Bl, streams=S, batch_split=split, handover_below=(args.handover if S > 1 and args.handover >= 0 else 1184), solver_handles=len(set(id(m) for m in dev_handles)),
                       pipeline_depth=args.pipeline,
                       note="value = problems_per_step x passes / seconds (max over ranks of the CUDA-event time)"),
            e2e=dict(value=e2e_value, unit=UNIT, h2d_bytes_per_step=total_per_step * (6 + ncoef) * 8,
                     d2h_bytes_per_step=total_per_step * (8 + 1) * 8 + 2 * total_per_step * 4, passes=n_e2e, seconds=e2e_max_s,
                     host_threads_per_gpu=T, calls_in_flight_per_gpu=S,
                     entry="b200mpc_solve_batch_async + b200mpc_wait, one pinned buffer set per solver handle" if T < S else "b200mpc_solve_batch",
                     p50_batch_latency_ms=1e3 * p50, p99_batch_latency_ms=1e3 * p99, latency_reps=len(lat),
                     latency_note="one host-buffer call at a time on one handle with library defaults, this rank's share of the batch"),
            lone_caller=dict(value=lone_value, unit=UNIT, handles=1, streams=1, batch_split=4, passes=n_lone,
                             avg_kernel_ms=lone_kernel_ms, launches_timed=lone_kern_n,
                             note="device-resident inputs, one solve call at a time on one handle (library defaults)"),
            gpu_launches=int(launches),
            clocks=dict(clocks, sm_mhz=cmhz if world > 1 else clocks.get("sm_mhz")), per_rank_ms_per_step=per_rank_ms, per_rank_sm_mhz=per_rank_mhz,
            roofline=dict(bound="fp64", achieved=achieved, peak=fp64_peak, unit="TFLOP/s", frac=achieved / fp64_peak if fp64_peak else None,
                          traffic=traffic, traffic_unit=prof.get("traffic_unit"),
                          hbm_achieved_gbs=traffic / (avg_kernel_ms * 1e-3) / 1e9 * (Bl / 65536.0) if traffic else None,
                          hbm_frac=(traffic / (avg_kernel_ms * 1e-3) / 1e9 * (Bl / 65536.0) / peaks["hbm_gbs"] if traffic and peaks.get("hbm_gbs") else None),
                          kernel=("mpc_{init,factor,forward,step,repack,coop}_kernel: all solver kernels of one step (one CUDA graph), first to last"
                                  if args.mode == "perpass" else "mpc_fused_kernel"),
                          avg_kernel_ms=avg_kernel_ms, avg_kernel_ms_one_stream=lone_kernel_ms,
                          frac_one_stream=lone_achieved / fp64_peak if fp64_peak else None,
                          executed_flop_per_step=prof.get("executed_flop_per_step"),
                          frac_executed=(prof["executed_flop_per_step"] * (Bl / 65536.0) / (avg_kernel_ms * 1e-3) / 1e12 / fp64_peak
                                         if prof.get("executed_flop_per_step") and fp64_peak else None),
                          executed_flop_source=prof.get("executed_flop_source"),
                          solver_mode=args.mode, streams=S, batch_split=split,
                          flop_per_step=flop_per_step, mean_ip_iters=mean_it,
                          peak_source="DFMA microbenchmark in this run (b200mpc_measure_fp64_peak); MEASURED_PEAKS.json has no FP64 figure",
                          hbm_peak_gbs=peaks.get("hbm_gbs"), algorithmic_io_bytes_per_solve=(6 + ncoef + 8 + 2) * 8,
                          note="SURVEY 8d classifies the solver as FP64 bound (intensity >> ridge, no tensor cores): achieved = F_iter(25)=62204 FLOP "
                               "(dense Riccati count) x mean iterations x problems / step device time, per GPU, over the measured DFMA peak.  The "
                               "kernels exploit the sparsity of the dynamics (frac_executed = FP64 FLOP actually executed, ncu) and in practice "
                               "sit between the issue and the HBM roof: hbm_frac = measured DRAM traffic of one step (ncu) / step time / measured "
                               "copy bandwidth"),
            solved_fraction=solved_fraction,
        )
        if multi:
            line["one_process_multi_gpu"] = multi
        if weak:
            line["weak_scaling"] = weak
        if world == 1 and not args.no_sweep:
            # BASELINE configs[4] in brief (bench_sweep.py has the full grid): other horizons at this batch size, 4
            # overlapped batches; N = 100 on one handle in pipelined mode (its tails are hundreds of iterations long)
            import bench_sweep
            sst, sfit = sets[0][0][:min(B, 65536)], sets[0][1][:min(B, 65536)]
            line["horizon_sweep"] = dict(
                note="solves/s at other horizons, same workload and batch size, device-resident inputs; 4 overlapped batches on 4 handles, "
                     "N = 100: 16 overlapped batches on ONE handle in pipelined mode (b200mpc_set_pipeline)",
                rows=[bench_sweep.run_point(mpcmod, torch, n_, B, sst, sfit, streams=s_, pipeline=p_, reps=r_, device=local)
                      for n_, s_, p_, r_ in ((10, 4, 0, 3), (50, 4, 0, 3), (100, 16, 16, 1))])
        if world == 1 and not args.no_cpu_baseline:
            st, cf = sets[0]
            line["cpu_baseline"] = {k: v for k, v in cpu_reference_rate(st[:8192], cf[:8192], args.cpu_per_core).items()}
        emit(line)
    lone.close()
    for m in mpcs:
        m.close()
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def claim_stdout():
    """Rank 0 must print exactly ONE line on stdout, but libraries write there too (NCCL's version banner comes from C
    code).  Everything written to fd 1 from here on goes to stderr; emit() writes the JSON line to the real stdout."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=65536, help="problems per step (the whole batch; sharded over the GPUs when --scaling strong)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong (default, BASELINE configs[3]): one --batch-problem batch per step sharded by index over the GPUs; "
                         "weak: every GPU solves its own --batch problems per step")
    ap.add_argument("--ref-per-core", type=int, default=200, help="--impl reference: solves per host core per step")
    ap.add_argument("--no-multi-leg", action="store_true", help="N > 1: skip the one-process b200mpc_solve_batch_multi leg")
    ap.add_argument("--no-weak-leg", action="store_true", help="N > 1: skip the weak-scaling figure")
    ap.add_argument("--workload", default="roadmap", choices=["roadmap", "line"])
    ap.add_argument("--latency-reps", type=int, default=100)
    ap.add_argument("--cpu-per-core", type=int, default=400, help="cpu_baseline: solves per host core in the sample (>= 2 s per core)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sweep", action="store_true", help="N = 1: skip the short horizon sweep (BASELINE configs[4]) appended to the line")
    ap.add_argument("--input-sets", type=int, default=4, help="distinct synthetic input batches cycled over the steps")
    ap.add_argument("--e2e-threads", type=int, default=0, help="host threads (one solver handle each) of the end-to-end leg (0 = auto)")
    ap.add_argument("--split", type=int, default=0, help="internal batch split of one solve call (0 = 1 with several streams, 4 with one)")
    ap.add_argument("--streams", type=int, default=0, help="solver handles / CUDA streams consecutive steps alternate between (0 = auto: 6 at 65 536 problems per GPU, up to 16 for smaller shards)")
    ap.add_argument("--handover", type=int, default=64, help="overlapped solver handles: occupied slots at which the cooperative kernel takes a batch's "
                    "tail over (b200mpc_set_handover; -1 = library default 1184, which suits one call at a time)")
    ap.add_argument("--pipeline", type=int, default=0, help="> 0: the overlapped streams of the device-timed region share ONE solver handle in pipelined mode "
                    "with this many tail contexts (b200mpc_set_pipeline) instead of one handle per stream")
    ap.add_argument("--pipeline-slots", type=int, default=0, help="problems a tail context holds (0 = max(1024, batch / 16))")
    ap.add_argument("--mode", default="perpass", choices=["perpass", "fused"], help="solver execution mode (include/b200mpc.h)")
    ap.add_argument("--rounds", type=int, default=0, help="per-pass mode: rounds before the fused finisher (0 = library default)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="--impl ours: write the results of the last timed step to DIR/<name>.npy (float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    claim_stdout()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
